"""Timing of the inner-product kernels (csrc/inner.cu) and of the host weight build (ops.spline_integral_weights).

    python dev/dev_inner_product_timing.py [--out FILE.json]

Cases: the streaming kernel (scrib200_inner_product, one complex scalar) at 1e5 x 77 and 1e6 x 285; the matrix kernel
(scrib200_inner_product_matrix) at P x Q = 512 x 512 and 4096 x 64 with N = 2048, n = 77; the host weights at N = 1e5 and
1e6.  Every device input is larger than the 126 MB L2, so each timed pass reads HBM.  CUDA events around R launches after a
warm-up; the FP64 denominator is cuBLAS DGEMM (6144^3, best of 5) measured in the same run, as bench.py does.  Prints the
card name and power limit with the numbers and one JSON document at the end."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

HBM_TBPS = 7.7   # B200 data sheet, per GPU


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as exc:          # the numbers are still printed, flagged as unattributed
        return {"name": "unknown", "power_limit": f"unknown ({exc})", "sm_clock_max": "unknown"}


def dgemm_tflops(torch, n=6144, reps=5):
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return 2.0 * n**3 / (best * 1e-3) / 1e12


def timed(torch, fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    from scri_b200 import _lib, ops

    if not torch.cuda.is_available():
        raise SystemExit("dev_inner_product_timing: no CUDA device")
    lib = _lib.load()
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['sm_clock_max']}", flush=True)
    res = {"card": info, "streaming": [], "matrix": [], "host_weights": []}
    dg = dgemm_tflops(torch)
    res["dgemm_tflops"] = dg
    print(f"cuBLAS DGEMM 6144^3: {dg:.2f} TFLOP/s", flush=True)
    gen = torch.Generator(device="cuda").manual_seed(0)

    def crand(*shape):
        return torch.randn(*shape, dtype=torch.complex128, device="cuda", generator=gen)

    for N, n, reps in [(100_000, 77, 50), (1_000_000, 285, 10)]:
        a, b = crand(N, n), crand(N, n)
        w = torch.rand(N, dtype=torch.float64, device="cuda", generator=gen)
        out = torch.empty(1, dtype=torch.complex128, device="cuda")
        ws = torch.empty(lib.scrib200_inner_product_workspace_bytes(N, n, 1), dtype=torch.uint8, device="cuda")
        st = _lib.stream_ptr()

        def run():
            _lib.check(lib.scrib200_inner_product(_lib.ptr(a), n, 0, 0, _lib.ptr(b), n, 0, 0, N, n, 1, _lib.ptr(w), 1, 0, _lib.ptr(out),
                                                  _lib.ptr(ws), ws.numel(), st), "inner_product")

        ms = timed(torch, run, reps)
        nbytes = 32.0 * N * n + 8.0 * N
        r = {"N": N, "n": n, "ms": ms, "TBps": nbytes / (ms * 1e-3) / 1e12, "frac_hbm": nbytes / (ms * 1e-3) / 1e12 / HBM_TBPS}
        res["streaming"].append(r)
        print(f"streaming {N} x {n}: {ms:.3f} ms, {r['TBps']:.2f} TB/s = {r['frac_hbm']:.2f} of {HBM_TBPS} TB/s", flush=True)
        del a, b

    N, n = 2048, 77
    for P, Q, reps in [(512, 512, 5), (4096, 64, 5)]:
        A, B = crand(P, N, n), crand(Q, N, n)
        w = torch.rand(N, dtype=torch.float64, device="cuda", generator=gen)
        G = torch.empty((P, Q), dtype=torch.complex128, device="cuda")
        ws = torch.empty(lib.scrib200_inner_product_matrix_workspace_bytes(P, Q, N, n), dtype=torch.uint8, device="cuda")
        st = _lib.stream_ptr()

        def run():
            _lib.check(lib.scrib200_inner_product_matrix(_lib.ptr(A), P, N * n, _lib.ptr(B), Q, N * n, N, n, _lib.ptr(w), _lib.ptr(G),
                                                         _lib.ptr(ws), ws.numel(), st), "inner_product_matrix")

        ms = timed(torch, run, reps)
        flops = 8.0 * P * Q * N * n            # real flops of the four-product form (2 per multiply-add)
        nbytes = 16.0 * (P + Q) * N * n
        tf = flops / (ms * 1e-3) / 1e12
        r = {"P": P, "Q": Q, "N": N, "n": n, "ms": ms, "TFLOPs": tf, "frac_dgemm": tf / dg,
             "hbm_floor_ms": nbytes / (HBM_TBPS * 1e12) * 1e3, "workspace_MB": ws.numel() / 1e6}
        res["matrix"].append(r)
        print(f"matrix {P} x {Q} (N={N}, n={n}): {ms:.3f} ms, {tf:.2f} TFLOP/s = {tf / dg:.2f} of DGEMM; "
              f"HBM floor {r['hbm_floor_ms']:.3f} ms", flush=True)
        del A, B

    rng = np.random.default_rng(1)
    for N in (100_000, 1_000_000):
        t = np.cumsum(rng.uniform(0.5, 1.5, N))
        ops.spline_integral_weights(t)
        best = 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            ops.spline_integral_weights(t)
            best = min(best, time.perf_counter() - t0)
        res["host_weights"].append({"N": N, "ms": best * 1e3})
        print(f"host weights N={N}: {best * 1e3:.1f} ms", flush=True)

    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
