"""Timing of the batched transform of psi2 (companions psi3 and psi4) against h on the same batch, at the shape of
BASELINE configs[2]: 4096 waveforms x 2048 steps, ell <= 8, supertranslation (ell <= 4) + rotation + boost, which puts
the grid at 25 x 25 points.

    python dev/dev_weyl_batch_timing.py [--batch 4096] [--out FILE.json]

Legs, each for h and for psi2 on the same time axis and transformation:
  device  parallel.transform_batch over the batch, held on the device in chunks of 512 waveforms (CUDA events around
          whole passes over the batch, after two warm-up passes);
  host    parallel.transform_batch_host from page-locked host memory at the default sub-batch (h: 512, psi2: 512 // 3 = 170)
          and at 64: the batch is 8 host blocks that share one page-locked block of 512 waveforms (and one result block),
          as bench.py's batch leg does (host clock around calls that end in a synchronise; best and mean of 3);
  mix     scrib200_weyl_mix_series alone with 3 fields in place (out = field 0, as the transform calls it) over
          512 x 2048 rows of 625 points (31 GB of operands, far beyond L2): (Q + 2) 16 bytes per element over the kernel
          time, against 7.7 TB/s.
Prints the card name and power limit with the numbers and one JSON document at the end."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM_TBPS = 7.7   # B200 data sheet, per GPU
N, CHUNK = 2048, 512


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as exc:          # the numbers are still printed, flagged as unattributed
        return {"name": "unknown", "power_limit": f"unknown ({exc})", "sm_clock_max": "unknown"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    import scri_b200 as sb
    from scri_b200 import _lib, _sf, parallel
    from scri_b200.plan import TransformPlan
    from scri_inputs import real_supertranslation

    if not torch.cuda.is_available():
        raise SystemExit("dev_weyl_batch_timing: no CUDA device")
    lib = _lib.load()
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['sm_clock_max']}", flush=True)
    B = args.batch
    assert B % CHUNK == 0
    kw = dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03])
    t = torch.linspace(0.0, 204.7, N, dtype=torch.float64, device="cuda")
    t_host = t.cpu().numpy()
    gen = torch.Generator(device="cuda").manual_seed(1234)

    def chunk(n):
        wf = torch.rand(CHUNK, 1, n, dtype=torch.float64, device="cuda", generator=gen) * 0.45 + 0.05
        c = torch.randn(CHUNK, 1, n, dtype=torch.complex128, device="cuda", generator=gen)
        return c * torch.exp(1j * wf * t[None, :, None])

    def layout(DT):
        s = abs(sb.SpinWeights[DT])
        return s, _sf.LM_total_size(s, 8)

    def host_modes(DT):
        s, n = layout(DT)
        return sb.WaveformModes(t=t_host.copy(), data=np.zeros((N, n), complex), ell_min=s, ell_max=8, frameType=sb.Inertial,
                                dataType=DT, r_is_scaled_out=True, m_is_scaled_out=True)

    plans = {
        "h": (TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **kw), [sb.h]),
        "psi2": (TransformPlan(0, 8, sb.psi2, r_is_scaled_out=True, psi3_modes=host_modes(sb.psi3), psi4_modes=host_modes(sb.psi4), **kw),
                 [sb.psi2, sb.psi3, sb.psi4]),
    }
    res = {"card": info, "batch": B, "n_times": N, "grid": None, "device": {}, "host": {}, "mix": None}
    for name, (plan, fields) in plans.items():
        res["grid"] = [plan.n_theta, plan.n_phi]
        data = [[chunk(layout(DT)[1]) for DT in fields] for _ in range(B // CHUNK)]

        def step():
            for d in data:
                parallel.transform_batch(plan, t, d[0], companions=d[1:] or None)

        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record()
        for _ in range(reps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res["device"][name] = {"ms_per_batch": ms, "us_per_waveform": 1e3 * ms / B, "chunk": CHUNK, "fields": len(fields)}
        print(f"device {name}: {ms:.1f} ms per {B} waveforms ({1e3 * ms / B:.1f} us per waveform, {len(fields)} fields)", flush=True)

        # end to end: one page-locked block of CHUNK waveforms per field, sent again for every block of the batch
        host_in = []
        for DT, d in zip(fields, data[0]):
            p = torch.empty(d.shape, dtype=torch.complex128, pin_memory=True)
            p.copy_(d)
            host_in.append(p.numpy())
        del data
        torch.cuda.empty_cache()
        n_blocks = B // CHUNK
        u, m = parallel.transform_batch(plan, t, torch.from_numpy(host_in[0][:1]).cuda(),
                                        companions=[torch.from_numpy(c[:1]).cuda() for c in host_in[1:]] or None)
        host_out = torch.empty((CHUNK, m.shape[1], m.shape[2]), dtype=torch.complex128, pin_memory=True).numpy()
        res["host"][name] = {}
        for sub in (None, 64):
            def e2e():
                parallel.transform_batch_host(plan, t_host, [host_in[0]] * n_blocks, sub_batch=sub, out=[host_out] * n_blocks,
                                              companions_host=[host_in[1:]] * n_blocks if len(fields) > 1 else None)

            for _ in range(2):
                e2e()
            torch.cuda.synchronize()
            times = []
            for _ in range(3):
                t0 = time.perf_counter()
                e2e()
                torch.cuda.synchronize()
                times.append(1e3 * (time.perf_counter() - t0))
            label = "default" if sub is None else str(sub)
            sub_used = sub if sub is not None else 512 // len(fields)
            res["host"][name][label] = {"sub_batch": sub_used, "ms_best": min(times), "ms_mean": float(np.mean(times)),
                                        "h2d_bytes": float(sum(c.nbytes for c in host_in) * n_blocks),
                                        "d2h_bytes": float(host_out.nbytes * n_blocks)}
            print(f"host {name} sub_batch {sub_used}: {min(times):.1f} ms best, {np.mean(times):.1f} ms mean per {B} waveforms",
                  flush=True)
        del host_in, host_out
        torch.cuda.empty_cache()
    for leg in ("device",):
        res[leg]["psi2_over_h"] = res[leg]["psi2"]["ms_per_batch"] / res[leg]["h"]["ms_per_batch"]
    res["host"]["psi2_over_h_default"] = res["host"]["psi2"]["default"]["ms_best"] / res["host"]["h"]["default"]["ms_best"]
    print(f"psi2 / h: device {res['device']['psi2_over_h']:.2f}, host (default sub-batches) {res['host']['psi2_over_h_default']:.2f}",
          flush=True)

    # the mixing kernel alone, in place, 3 fields (psi2 + psi3 + psi4): 512 x 2048 rows x 625 points
    plan = plans["psi2"][0]
    G, S = plan.G, CHUNK
    Fs = [torch.randn((S * N, G), dtype=torch.complex128, device="cuda", generator=gen) for _ in range(3)]
    ptrs = (ctypes.c_void_p * 3)(*[f.data_ptr() for f in Fs])
    cf = (ctypes.c_double * 3)(1.0, 3.0, 3.0)

    def mix():
        _lib.check(lib.scrib200_weyl_mix_series(ptrs, cf, 3, _lib.ptr(t), N, S, G, _lib.ptr(plan.d_alpha), _lib.ptr(plan.d_mixA),
                                                _lib.ptr(plan.d_mixC), _lib.ptr(plan.d_mixscale), None, _lib.ptr(Fs[0]),
                                                _lib.stream_ptr()), "weyl_mix_series")

    for _ in range(2):
        mix()
    torch.cuda.synchronize()
    reps = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        mix()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    nbytes = (3 + 1) * 16.0 * S * N * G
    tbps = nbytes / (ms * 1e-3) / 1e12
    res["mix"] = {"n_series": S, "n_times": N, "G": G, "fields": 3, "ms": ms, "bytes": nbytes, "TBps": tbps, "frac_hbm": tbps / HBM_TBPS}
    print(f"weyl_mix_series {S} x {N} x {G}, 3 fields in place: {ms:.3f} ms, {tbps:.2f} TB/s = {tbps / HBM_TBPS:.2f} of {HBM_TBPS} TB/s",
          flush=True)

    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
