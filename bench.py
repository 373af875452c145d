#!/usr/bin/env python
"""bench.py - mode-timesteps/s through WaveformModes.transform (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n-times T] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): fake_precessing_waveform, ell 2..8 (77 modes), ~1e5 time steps,
transform(supertranslation with ell<=4, frame_rotation, boost_velocity) -> working band limit 12, 25x25 grid.
A "step" is one pass of the whole path (synthesis -> spline remap -> analysis) over that waveform.
For N > 1 GPUs every rank runs its own waveform of that size (batch of N waveforms sharded by waveform
index, no data-path collective): weak scaling; value = total mode-timesteps of all ranks / max-over-ranks time.

  value : device-resident - inputs and the plan's tables already in HBM, CUDA-event time of plan.run()
  e2e   : the public call w.transform(**kwargs) on host numpy arrays: plan construction, H2D, kernels, D2H
  --impl reference : the reference's CPU algorithm (oracle/, a port: the reference itself cannot be
          imported here) on a bounded time-slice of the same waveform, grid points spread over all host cores.
  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned (output times and modes,
          a fixed sample of DUMP_ROWS output times) as float64 .npy files, so that two builds can be compared output
          for output: the inputs are the same from run to run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

_JSON_FD = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line at init when
    NCCL_DEBUG is set), so file descriptor 1 is pointed at stderr for the whole run and the JSON line alone goes to the
    original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line, default=float) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, data)


METRIC = "mode-timesteps/sec through WaveformModes.transform (ell_max=8)"
UNIT = "mode-timesteps/s"


def transformation_kwargs():
    from scri_inputs import real_supertranslation

    return dict(
        supertranslation=real_supertranslation(4, seed=123, scale=1e-2),
        frame_rotation=[1.0, 2.0, 3.0, 4.0],
        boost_velocity=[0.01, 0.02, 0.03],
    )


def make_workload(n_times, corotating_only=False):
    """(t, data[n_times, 77], frame) host arrays of the config-2 waveform (inertial frame needs the GPU)."""
    import scri_b200 as sb

    dt = 0.1
    w = sb.sample_waveforms.fake_precessing_waveform(t_0=-20.0, t_1=-20.0 + dt * (n_times - 1), dt=dt, ell_max=8, inertial=not corotating_only)
    return w


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax = float(parts[1])
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_ROWS = 32768   # output times kept by --dump-outputs: 32768 x 77 modes x 16 B = 41 MB, under 64 MB at any --n-times


def dump_outputs(out_dir, t, data):
    """DIR/t.npy: output times; DIR/data.npy: modes as (time, mode, re/im); DIR/rows.npy: which output times these are
    (all of them when there are at most DUMP_ROWS, else a sorted sample drawn with a fixed seed)."""
    t, data = t.cpu().numpy(), data.cpu().numpy()
    n = t.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS), replace=False))
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "t.npy"), t[rows])
    np.save(os.path.join(out_dir, "data.npy"), np.ascontiguousarray(data[rows]).view(np.float64).reshape(rows.size, *data.shape[1:], 2))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


def measure_dgemm_peak(torch, n=6144, reps=5):
    """cuBLAS DGEMM throughput (TFLOP/s) - the FP64 denominator MEASURED_PEAKS.json does not carry."""
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


def cpu_baseline_sample(w_t, w_data, kw, n_sample, workers=1):
    """Oracle (CPU port of the reference algorithm) on the first n_sample time steps; returns (value, seconds, n_out)."""
    from oracle import scri_ref as R

    Wo = R.Modes(t=w_t[:n_sample].copy(), data=w_data[:n_sample].copy())
    t0 = time.perf_counter()
    if workers > 1:
        out = oracle_transform_parallel(Wo, kw, workers)
    else:
        out = R.transform(Wo, **kw)
    dt = time.perf_counter() - t0
    return 77.0 * n_sample / dt, dt, out.t.shape[0]


def _spline_columns(args):
    from scipy import interpolate

    t, kc, al, cols_re, cols_im, uprm = args
    out = np.empty((uprm.shape[0], cols_re.shape[1]), dtype=complex)
    for c in range(cols_re.shape[1]):
        x = kc[c] * (t - al[c])
        out[:, c] = interpolate.InterpolatedUnivariateSpline(x, cols_re[:, c])(uprm) + 1j * interpolate.InterpolatedUnivariateSpline(x, cols_im[:, c])(uprm)
    return out


def oracle_transform_parallel(Wo, kw, workers):
    """The oracle's transform with the per-grid-point spline loop (waveform_grid.py:576-588) spread over processes.

    Same arithmetic per grid point as oracle.scri_ref.from_modes; everything else is the oracle itself.
    """
    import multiprocessing as mp

    from oracle import scri_ref as R
    from oracle import sf as osf

    g, inter = R.from_modes(R.Modes(t=Wo.t[:8].copy(), data=Wo.data[:8].copy()), return_intermediates=True, **dict(kw))
    # synthesis for the full sample with the oracle's own tables
    SW = inter["SWSH_j_k"]
    kc, al = inter["kconformal"], inter["alpha"]
    nth, nph = kc.shape
    (st, ell_st, L, _, _, bv, beta, gamma, _, R_j_k, _) = R.process_transformation_kwargs(Wo.ell_max, **dict(kw))
    f = np.tensordot(Wo.data, SW[:, :, osf.LM_index(Wo.ell_min, -Wo.ell_min, 0) : osf.LM_index(Wo.ell_max, Wo.ell_max, 0) + 1], axes=([1], [2]))
    deriv = 2 * osf.ethbar_GHP(osf.ethbar_GHP(st, 0, 0), -1, 0)
    f -= np.tensordot(deriv, SW[:, :, : (ell_st + 1) ** 2], axes=([0], [2]))[None]
    f *= (kc**Wo.conformal_weight)[None]
    tt = osf.constant_from_ell_0_mode(st[0]).real
    uprm_i = (1 / gamma) * (Wo.t - tt)
    umin = (kc * (Wo.t[0] - al)).max()
    umax = (kc * (Wo.t[-1] - al)).min()
    uprm = uprm_i[(uprm_i >= umin) & (uprm_i <= umax)]
    f2 = f.reshape(f.shape[0], -1)
    G = f2.shape[1]
    bounds = np.linspace(0, G, workers + 1).astype(int)
    jobs = [(Wo.t, kc.ravel()[a:b], al.ravel()[a:b], np.ascontiguousarray(f2[:, a:b].real), np.ascontiguousarray(f2[:, a:b].imag), uprm) for a, b in zip(bounds[:-1], bounds[1:]) if b > a]
    with mp.get_context("fork").Pool(workers) as pool:
        parts = pool.map(_spline_columns, jobs)
    grid = np.concatenate(parts, axis=1)
    return R.to_modes(R.Grid(t=uprm, data=grid, n_theta=nth, n_phi=nph), Wo.ell_max)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kw = transformation_kwargs()
    n_sample = args.ref_sample
    import scri_b200 as sb  # host-only generator (corotating-frame data, rotated with the oracle)
    from oracle import scri_ref as R

    wc = make_workload(n_sample, corotating_only=True)
    Wo = R.Modes(t=wc.t.copy(), data=wc.data.copy(), frame=wc.frame.copy(), frameType=R.Corotating)
    R.to_inertial_frame(Wo)
    cores = os.cpu_count() or 1
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        oracle_transform_parallel(R.Modes(t=Wo.t, data=Wo.data), kw, cores)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = 77.0 * n_sample / (ms * 1e-3)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"configs[1]: fake_precessing_waveform ell_max=8, transform(supertranslation ell<=4 + rotation + boost); bounded sample of {n_sample} time steps per step", "n_times": n_sample, "n_modes": 77, "grid": "25x25"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"first {n_sample} time steps of the configs[1] waveform, oracle/ port of scri's algorithm (scipy FITPACK splines), spline loop over {cores} processes"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def extra_batch(args, torch, dist, world, rank, kw):
    """BASELINE configs[2] next to the headline line: 4096 random-mode waveforms (ell 2..8, 2048 steps each), one shared
    transformation, the batch sharded by waveform index over the ranks (STRONG scaling, no data-path collective).
    Two legs: device-resident (plan.run_batch over the rank's shard) and end to end from pinned host memory
    (parallel.transform_batch_host: H2D, kernels and D2H of every sub-batch inside the timed region)."""
    import scri_b200 as sb
    from scri_b200 import parallel
    from scri_b200.plan import TransformPlan

    B, N, n, sub = args.batch, 2048, 77, 512
    lo, hi = parallel.shard_range(B, rank, world)
    plan = TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **kw)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    t = torch.linspace(0.0, 204.7, N, dtype=torch.float64, device="cuda")
    chunks = []
    for b0 in range(lo, hi, sub):
        bn = min(sub, hi - b0)
        wf = torch.rand(bn, 1, n, dtype=torch.float64, device="cuda", generator=g) * 0.45 + 0.05
        c = torch.randn(bn, 1, n, dtype=torch.complex128, device="cuda", generator=g)
        chunks.append(c * torch.exp(1j * wf * t[None, :, None]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        n_out = 0
        for d in chunks:
            up, out = plan.run_batch(t, d)
            n_out = up.shape[0]
        return n_out

    steps = max(3, min(args.steps, 5))
    for _ in range(3):
        n_out = step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        n_out = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / steps
    # end to end: the rank's shard lives in pinned host memory as ONE sub-batch worth of waveforms that is sent again for
    # every sub-batch of the shard (same bytes over PCIe as a full host copy of the shard, a twelfth of the host RAM)
    host_in = torch.empty((min(sub, hi - lo), N, n), dtype=torch.complex128, pin_memory=True)
    host_in.copy_(chunks[0][: host_in.shape[0]])
    torch.cuda.synchronize()
    t_host = t.cpu().numpy()
    shard = hi - lo
    reps = -(-shard // host_in.shape[0])
    host_out = torch.empty((host_in.shape[0], int(n_out), n), dtype=torch.complex128, pin_memory=True)

    def e2e_step():
        # the shard as `reps` host blocks flowing through one pipeline (the same pinned blocks each time, see above)
        sizes = [min(host_in.shape[0], shard - r * host_in.shape[0]) for r in range(reps)]
        u, res = parallel.transform_batch_host(plan, t_host, [host_in.numpy()[:nb] for nb in sizes], sub_batch=sub // 8,
                                               out=[host_out[:nb] for nb in sizes])
        return u

    for _ in range(2):
        e2e_step()
    barrier()
    times = []
    for _ in range(3):
        t0 = time.perf_counter()
        e2e_step()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    e2e_ms = 1e3 * float(np.mean(times))
    tms = torch.tensor([ms, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(tms[0]), float(tms[1])
    del chunks
    torch.cuda.empty_cache()
    units = float(n) * N * B
    return {
        "workload": f"configs[2]: batch of {B} random-mode waveforms, ell 2..8 (77 modes), {N} steps each, one shared transformation; sharded by waveform index (sub-batches of {sub}), no collective",
        "scaling": "strong", "value": units / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "n_out": int(n_out),
        "e2e": {"value": units / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(shard) * N * n * 16 * world, "d2h_bytes_per_step": int(shard) * int(n_out) * n * 16 * world,
                "note": f"host arrays in pinned memory ({sub} waveforms per call of parallel.transform_batch_host, sub-batches of {sub // 8} double-buffered on three streams, one spline preparation for the whole batch); H2D, kernels and D2H of every sub-batch inside the timed region"},
    }


def extra_timeshard(args, torch, dist, world, rank, kw, w):
    """BASELINE configs[1] as ONE series sharded by TIME over the ranks (strong scaling): parallel.sharded_transform, whose
    only data-path communication is the point-to-point halo exchange of the input modes plus a 4-scalar all_gather; the two
    are timed separately with CUDA events."""
    from scri_b200 import ops, parallel
    from scri_b200.plan import TransformPlan

    N = w.t.shape[0]
    lo, hi = parallel.shard_range(N, rank, world)
    t_d = ops.to_device(np.ascontiguousarray(w.t[lo:hi]))
    a_d = ops.to_device(np.ascontiguousarray(w.data[lo:hi]))
    plan = TransformPlan(w.ell_min, w.ell_max, w.dataType, r_is_scaled_out=w.r_is_scaled_out, **kw)
    halo = parallel.transform_halo(plan, float(w.t[lo]), float(w.t[hi - 1]), float(np.diff(w.t).min()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    for _ in range(3):
        u, m = parallel.sharded_transform(plan, t_d, a_d)
    barrier()
    steps = max(3, min(args.steps, 10))
    total = ag = p2p = 0.0
    for _ in range(steps):
        flush.zero_()
        barrier()
        tm = {}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        u, m = parallel.sharded_transform(plan, t_d, a_d, timings=tm)
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
        ag += tm["all_gather_begin"].elapsed_time(tm["all_gather_end"])
        p2p += tm["halo_begin"].elapsed_time(tm["halo_end"])
    tms = torch.tensor([total / steps, ag / steps, p2p / steps], dtype=torch.float64, device="cuda")
    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    n_out = torch.tensor([u.shape[0]], dtype=torch.int64, device="cuda")
    dist.all_reduce(n_out)
    ms = float(tms[0])
    return {
        "workload": f"configs[1] as one series of {N} steps sharded by time over {world} rank(s): halo of {halo} input samples per boundary exchanged point-to-point (NCCL), 4-scalar all_gather, no other collective",
        "scaling": "strong", "value": float(w.n_modes) * N / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "halo_samples": int(halo),
        "all_gather_4_scalars_ms": float(tms[1]), "halo_p2p_ms": float(tms[2]), "n_out": int(n_out[0]),
        "halo_bytes_per_boundary": int(halo) * (int(w.n_modes) * 16 + 8) * 2,
    }


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import scri_b200 as sb
    from scri_b200 import _lib, ops
    from scri_b200.plan import TransformPlan

    kw = transformation_kwargs()
    N = args.n_times
    w = make_workload(N)   # every rank builds the same-size waveform (its own unit of the batch)
    n_modes = w.n_modes
    plan = TransformPlan(w.ell_min, w.ell_max, w.dataType, r_is_scaled_out=True, **kw)
    t_d = ops.to_device(w.t)
    a_d = ops.to_device(w.data)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def staged_step(hold_cycles=0):
        # same calls as TransformPlan.run(), with events between the stages.  hold_cycles > 0 parks the stream on a spin
        # kernel first, so that the host has queued the whole step before the first stage starts: the intervals between
        # the events are then kernel time only, whatever the host's launch rate is
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        if hold_cycles:
            torch.cuda._sleep(int(hold_cycles))
        ev[0].record()
        F = plan.synthesize(a_d)
        ev[1].record()
        prep = plan.prepare(t_d, overlapped=True, after=ev[0], speculate=True)   # spline factor table, u', retained block: 4 tiny
        torch.cuda.current_stream().wait_event(prep.done)        # kernels on a side stream, running under the synthesis GEMM
        ev[2].record()
        up = prep.uprm
        if plan.tile:
            grid = plan.remap_tiled(t_d, F, up, prep)
            ev[3].record()
            m = plan.analyze_tiled(grid, up.shape[0])
        else:
            grid = plan.remap(t_d, F, up, prep)
            ev[3].record()
            m = plan.analyze(grid)
        ev[4].record()
        assert prep.verify()       # the retained block assumed from the previous step (same time axis) is what the kernels found
        return ev, up, m

    # ---- device-resident value.  Two loops over the same kernels: (1) the step as ONE CUDA-graph launch
    # (TransformPlan.capture) - this is `value`: the host is off the critical path, so a busy host cannot put gaps between
    # the kernels; (2) the eager step with events between the stages, for the per-kernel split and the roofline of the
    # dominant kernel: each eager step is queued behind a ~10 ms spin kernel, so that its event intervals hold kernel time
    # and no launch gaps even when the host launches slowly (seen on ~1 box in 3: eager steps of 3-4 ms over 2.3 ms of kernels).
    for _ in range(args.warmup):
        staged_step()
    barrier()
    captured = None
    try:
        captured = plan.capture(t_d, a_d)
        for _ in range(args.warmup):
            captured.replay()
        torch.cuda.synchronize()
        assert captured.verify()
    except Exception as exc:          # no graph: the eager loop below provides the value
        sys.stderr.write(f"[rank {rank}] CUDA-graph capture of the step failed ({type(exc).__name__}: {exc}); timing the eager step\n")
        captured = None
    barrier()
    # the collector stays off inside the timed regions, as in timeit: a generation-2 sweep of a process that has torch and
    # scipy loaded takes 40-120 ms and, landing in the middle of one step's launches, was charged to that step's kernels
    import gc

    gc.collect()
    gc.disable()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    per_kernel = np.zeros(4)
    eager_ms = 0.0
    n_out = 0
    n_eager = args.steps if captured is None else max(3, min(args.steps, 50))
    barrier()
    wall0 = time.perf_counter()
    for _ in range(n_eager):
        flush.fill_(1)   # L2 flush between timed iterations (outside the per-step event pairs)
        ev, up, m = staged_step(hold_cycles=2e7)
        torch.cuda.synchronize()
        eager_ms += ev[0].elapsed_time(ev[4])
        per_kernel += [ev[i].elapsed_time(ev[i + 1]) for i in range(4)]
        n_out = up.shape[0]
    launches_per_step = (_lib.launch_count() - launches0) // n_eager
    per_kernel /= n_eager
    eager_ms /= n_eager
    step_launch = "one CUDA-graph launch per step (TransformPlan.capture)" if captured is not None else "eager"
    if captured is not None:
        total_ms = 0.0
        for _ in range(args.steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            up, m = captured.replay()
            e1.record()
            torch.cuda.synchronize()
            total_ms += e0.elapsed_time(e1)
        assert captured.verify()
        ms_step = total_ms / args.steps
    else:
        ms_step = eager_ms
    barrier()
    wall = time.perf_counter() - wall0
    launches = launches_per_step * args.steps      # kernels of ours per step (counted in the eager loop) x timed steps
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, up, m)     # the last timed step's (u', modes'), before anything else runs

    # ---- e2e: the public API on host arrays (plan construction + H2D + kernels + D2H inside the timed region)
    # warm-up: the pinned-host caching allocator needs a few calls before result buffers are recycled
    out = None
    gc.enable()
    for _ in range(max(args.warmup, 5)):
        out = w.transform(**kw)
    barrier()
    gc.collect()
    gc.disable()
    def e2e_loop():
        times = []
        for _ in range(max(3, min(args.steps, 10))):
            t0 = time.perf_counter()
            o = w.transform(**kw)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        return times, o

    # (a) the modes in an ordinary numpy array: the library page-locks it in place at its second sighting (warm-up above).
    # (`out` is dropped first: the loop holds one result while the next is produced - a third live result would need a third
    # page-locked block, i.e. a 60-80 ms cudaHostAlloc inside the timed region)
    out = None
    pageable_times, out = e2e_loop()
    # (b) the modes in page-locked host memory from the start (the contract's "from pinned host memory"): the headline e2e
    pageable_data = w.data
    pinned_block = torch.empty(w.data.shape, dtype=torch.complex128, pin_memory=True)
    pinned_view = pinned_block.numpy()
    pinned_view[...] = w.data
    w.data = pinned_view
    gc.enable()
    for _ in range(3):
        out = w.transform(**kw)
    out = None
    barrier()
    gc.collect()
    gc.disable()
    e2e_times, out = e2e_loop()
    w.data = pageable_data
    e2e_ms = 1e3 * float(np.mean(e2e_times))
    e2e_pageable_ms = 1e3 * float(np.mean(pageable_times))
    gc.enable()
    sys.stderr.write(f"[rank {rank}] e2e per call (ms), pinned input: " + " ".join(f"{1e3 * x:.2f}" for x in e2e_times) + "\n")
    sys.stderr.write(f"[rank {rank}] e2e per call (ms), numpy input (registered in place): " + " ".join(f"{1e3 * x:.2f}" for x in pageable_times) + "\n")
    h2d = w.t.nbytes + w.data.nbytes
    d2h = out.t.nbytes + out.data.nbytes

    # ---- what the host link alone allows: the same bytes (modes up, modes' down) as two bare DMAs on two streams, no
    # kernels, all ranks at once.  On a multi-GPU box the ranks share the host's PCIe fabric and memory controllers, so
    # this floor - not the kernels - is what e2e is measured against as N grows.
    copy_ms = None
    try:
        up_src = torch.empty(int(np.asarray(w.data).nbytes), dtype=torch.uint8, pin_memory=True)
        down_dst = torch.empty(int(out.data.nbytes + out.t.nbytes), dtype=torch.uint8, pin_memory=True)
        up_src.fill_(1), down_dst.fill_(1)
        d_up = torch.empty(up_src.numel(), dtype=torch.uint8, device="cuda")
        d_down = torch.ones(down_dst.numel(), dtype=torch.uint8, device="cuda")
        s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()
        reps = []
        for _ in range(6):
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s_up):
                d_up.copy_(up_src, non_blocking=True)
            with torch.cuda.stream(s_down):
                down_dst.copy_(d_down, non_blocking=True)
            torch.cuda.synchronize()
            reps.append((time.perf_counter() - t0) * 1e3)
        copy_ms = float(np.mean(reps[1:]))
        del up_src, down_dst, d_up, d_down
    except Exception as exc:
        sys.stderr.write(f"[rank {rank}] copy-only floor not measured ({type(exc).__name__}: {exc})\n")
    barrier()
    tms = torch.tensor([ms_step, e2e_ms, copy_ms if copy_ms is not None else 0.0, e2e_pageable_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_step_max, e2e_ms_max, e2e_pageable_ms_max = float(tms[0]), float(tms[1]), float(tms[3])
    copy_ms_max = float(tms[2]) if copy_ms is not None else None
    units = float(n_modes) * N * world
    value = units / (ms_step_max * 1e-3)
    e2e_value = units / (e2e_ms_max * 1e-3)

    # ---- what north_star asks of the 1 -> 8 GPU runs besides the headline line (extra keys of the same JSON line)
    extras = {}
    G, grid_str = plan.G, f"{plan.n_theta}x{plan.n_phi}"
    if not args.no_extras:
        del plan, a_d, flush, captured
        torch.cuda.empty_cache()
        try:
            extras["batch_config2"] = extra_batch(args, torch, dist, world, rank, kw)
        except Exception as exc:   # the headline line must survive a failure here
            extras["batch_config2"] = {"error": f"{type(exc).__name__}: {exc}"}
        try:
            if not dist.is_initialized():
                os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
                os.environ.setdefault("MASTER_PORT", str(29500 + os.getpid() % 2000))
                dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", local_rank))
            extras["timeshard_config1"] = extra_timeshard(args, torch, dist, world, rank, kw, w)
        except Exception as exc:
            extras["timeshard_config1"] = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        peaks, peak_kind = measured_peaks()
        # dominant kernel by time decides which roofline is quoted; all three are listed under "kernels"
        dgemm_tf = measure_dgemm_peak(torch)
        synth_flops = 8.0 * n_modes * G * N
        remap_bytes = 32.0 * G * N          # read F (16 G) + write grid' (16 G) per time step
        ana_bytes = (16.0 * G + 16.0 * n_modes) * n_out
        kern = {
            "swsh_synth_dmma": {"ms": per_kernel[0], "bound": "tensor(fp64)", "achieved_tflops": synth_flops / (per_kernel[0] * 1e-3) / 1e12},
            "spline_prepare(factor table, u', retained block; side stream, overlapped with the synthesis)": {"ms_exposed_on_main_stream": per_kernel[1]},
            "spline_tile(spline_remap)": {"ms": per_kernel[2], "bound": "hbm", "achieved_gbs": remap_bytes / (per_kernel[2] * 1e-3) / 1e9},
            "map2salm_tiled": {"ms": per_kernel[3], "bound": "hbm", "achieved_gbs": ana_bytes / (per_kernel[3] * 1e-3) / 1e9},
        }
        if per_kernel[2] >= per_kernel[0]:
            ach = kern["spline_tile(spline_remap)"]["achieved_gbs"]
            roof = {"kernel": "spline_tile_kernel<0, 320>", "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": ach / peaks["hbm_gbs"], "traffic": None, "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peak_kind})",
                    "algorithmic_bytes_per_launch": remap_bytes}
        else:
            ach = kern["swsh_synth_dmma"]["achieved_tflops"]
            roof = {"kernel": "swsh_synth3m_kernel<3>", "bound": "tensor", "achieved": ach, "peak": dgemm_tf, "unit": "TFLOP/s",
                    "frac": ach / dgemm_tf, "traffic": None,
                    "peak_source": "cuBLAS DGEMM 6144^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                    "algorithmic_flops_per_launch": synth_flops,
                    "note": "algorithmic flops = 8 n G per time step (SURVEY 8d, a complex GEMM); the kernel forms the complex product with three real multiplications, so the tensor cores execute 6 n G"}
        # DRAM traffic per launch: dram__bytes_read.sum + dram__bytes_write.sum of the same kernels at this size from the round's
        # committed `ncu --set full` capture (profiles/r02_traffic.json, made with dev/dev_ncu_traffic.py; ncu cannot run
        # inside a timed region)
        try:
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                traffic = json.load(f)
            names = {"swsh_synth_dmma": "swsh_synth3m_kernel<3>", "spline_tile(spline_remap)": "spline_tile_kernel<0, 320>",
                     "map2salm_tiled": "map2salm_persist_kernel<1>"}
            for kname, ncu_name in names.items():
                if ncu_name in traffic:
                    kern[kname]["dram_bytes_per_launch(ncu, profiles/r02_ncu_summary.md)"] = traffic[ncu_name]["dram_bytes_per_launch"]
            roof["traffic"] = traffic.get(roof["kernel"], {}).get("dram_bytes_per_launch")
            roof["traffic_source"] = "dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full, profiles/r02_ncu_summary.md (N = 1e5 capture)"
        except Exception:
            pass
        # CPU baseline: oracle port, single thread + BLAS, bounded sample
        cpu_cores = 1
        cval, csec, _ = cpu_baseline_sample(w.t, w.data, kw, args.cpu_sample, workers=1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step_max, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {
                "workload": "configs[1]: fake_precessing_waveform ell_max=8 (77 modes), transform(supertranslation ell<=4 + frame_rotation + boost_velocity), 25x25 grid; one such waveform per GPU (batch sharded by waveform index)",
                "n_times": N, "n_out": n_out, "n_modes": n_modes, "grid": grid_str,
                "l2": "explicit 256 MiB L2 flush between timed iterations; intermediates (2 x 1 GB) exceed L2",
                "gc": "Python's cyclic collector disabled inside the timed regions (as timeit does)",
            },
            "roofline": roof, "kernels": kern, "fp64_dgemm_tflops_measured": dgemm_tf,
            # SURVEY.md 8(d): 5.4e10 flop per configs[1] transform (synthesis 3.85e10 + spline 0.56e10 + separable analysis ~1e10);
            # the north_star target is 60 % of the FP64 tensor roofline for the whole step
            "whole_transform": {"algorithmic_flops": 5.4e10 * N / 1e5, "achieved_tflops": 5.4e10 * N / 1e5 / (ms_step_max * 1e-3) / 1e12,
                                "frac_of_measured_dgemm": 5.4e10 * N / 1e5 / (ms_step_max * 1e-3) / 1e12 / dgemm_tf, "target_frac": 0.60},
            "cpu_baseline": {"value": cval, "unit": UNIT, "cores": cpu_cores, "kind": "port",
                             "sample": f"first {args.cpu_sample} time steps of the same waveform through oracle/ (port of scri's algorithm, scipy FITPACK splines; reference packages not installable here), {csec:.1f} s; host has {os.cpu_count()} cores"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms_max,
                    "input": "modes in page-locked host memory (numpy view of a pinned block); result in pinned memory from the library's pool",
                    "numpy_input_ms_per_step": e2e_pageable_ms_max,
                    "numpy_input_note": "the same call on an ordinary numpy array, which the library page-locks in place (cudaHostRegister) at its second sighting",
                    "copy_only_ms_per_step": copy_ms_max,
                    "copy_only_note": "the same H2D + D2H bytes as two bare DMAs (pinned memory, two streams, no kernels), all ranks at once, max over ranks: what the host link allows at this N"},
            "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": wall,
            "step_launch": step_launch,
            "eager_ms_per_step": eager_ms,
        }
        line.update(extras)
        emit(line)
    if dist.is_initialized():
        dist.destroy_process_group()


def run_batch_workload(args):
    """BASELINE configs[2]: a batch of random-mode waveforms (l <= 8, 2048 steps each) sharing one BMS transformation,
    sharded by waveform index over the ranks (strong scaling: the batch is fixed).  Optional workload, not the
    default bench line; device-resident only (the reference has no batched call to mirror end to end)."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import scri_b200 as sb
    from scri_b200 import _lib, parallel
    from scri_b200.plan import TransformPlan

    kw = transformation_kwargs()
    B, N, n = args.batch, 2048, 77
    lo, hi = parallel.shard_range(B, rank, world)
    plan = TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **kw)
    g = torch.Generator(device="cuda").manual_seed(1234 + rank)
    t = torch.linspace(0.0, 204.7, N, dtype=torch.float64, device="cuda")
    sub = 512
    chunks = []
    for b0 in range(lo, hi, sub):
        bn = min(sub, hi - b0)
        w = torch.rand(bn, 1, n, dtype=torch.float64, device="cuda", generator=g) * 0.45 + 0.05
        c = torch.randn(bn, 1, n, dtype=torch.complex128, device="cuda", generator=g)
        chunks.append(c * torch.exp(1j * w * t[None, :, None]))

    def step():
        n_out = 0
        for d in chunks:
            up, out = plan.run_batch(t, d)
            n_out = up.shape[0]
        return n_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        n_out = step()
    e1.record()
    barrier()
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1) / args.steps
    tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms[0])
    if rank == 0:
        line = {
            "metric": METRIC, "value": float(n) * N * B / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"configs[2]: batch of {B} random-mode waveforms, ell 2..8 (77 modes), {N} steps each, one shared transformation (supertranslation ell<=4 + rotation + boost); sharded by waveform index, sub-batches of {sub}",
                       "n_out": n_out, "grid": f"{plan.n_theta}x{plan.n_phi}",
                       "l2": "every sub-batch streams > 20 GB of intermediates: far beyond L2"},
            "e2e": None, "gpu_launches": int(launches), "clocks": clocks,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_product_workload(args):
    """BASELINE configs[3] (AsymptoticBondiData ell_max = 32, 1e5 steps): the mode product sigma x d/dt(bar sigma) of the
    mass aspect / supermomentum (scri/asymptotic_bondi_data/bms_charges.py:40,243) on the 129 x 129 working grid through
    the fused separable kernel K9 (scrib200_modes_product).  The time steps are independent: sharded by time over the
    ranks with no collective (strong scaling).  Optional workload, not the default bench line."""
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from scri_b200 import _lib, _product, ops, parallel

    L, N = 32, args.n_times
    n = (L + 1) ** 2
    lo, hi = parallel.shard_range(N, rank, world)
    g = torch.Generator(device="cuda").manual_seed(99 + rank)
    a = torch.view_as_complex(torch.randn((hi - lo, n, 2), dtype=torch.float64, device="cuda", generator=g))
    b = torch.view_as_complex(torch.randn((hi - lo, n, 2), dtype=torch.float64, device="cuda", generator=g))
    a[:, :4] = 0
    b[:, :4] = 0
    tb = _product.product_tables(2, 0, L, -2, 0, L, 2 * 2 * L + 1, 2 * 2 * L + 1, L)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step():
        return ops.modes_product(a, 2, 0, L, b, -2, 0, L, 2 * 2 * L + 1, 2 * 2 * L + 1, L)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    dgemm = measure_dgemm_peak(torch) if rank == 0 else None
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = _lib.launch_count()
    total = 0.0
    barrier()
    for _ in range(args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    barrier()
    launches = _lib.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    ms = total / args.steps
    tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms[0])
    if rank == 0:
        # CPU baseline: the reference's chain (salm2map x 2, product, map2salm) in the oracle port, a few steps
        import time as _time
        from oracle import abd_ref

        ns = 8
        ah, bh = a[:ns].cpu().numpy(), b[:ns].cpu().numpy()
        t0 = _time.perf_counter()
        ref = abd_ref.grid_multiply(ah, 2, bh, -2, working_ell_max=2 * L, output_ell_max=L)
        cpu_s = _time.perf_counter() - t0
        out = step()[:ns].cpu().numpy()
        err = float(np.abs(out - ref).max() / np.abs(ref).max())
        flops = tb.flops_per_step * (hi - lo)
        # the other half of configs[3]: SWSH grid round trip of one l <= 32 field on its 65 x 65 grid (separable salm2map / map2salm)
        nrt = min(hi - lo, 50_000)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        ops.map2salm(ops.salm2map(a[:64], 2, L, 2 * L + 1, 2 * L + 1), 2, L, 2 * L + 1, 2 * L + 1)
        flush.zero_()
        e0.record()
        grid = ops.salm2map(a[:nrt], 2, L, 2 * L + 1, 2 * L + 1)
        e1.record()
        back = ops.map2salm(grid, 2, L, 2 * L + 1, 2 * L + 1)
        e2.record()
        torch.cuda.synchronize()
        rt_err = float((back - a[:nrt]).abs().max() / a[:nrt].abs().max())
        round_trip = {"n_times": nrt, "grid": f"{2 * L + 1}x{2 * L + 1}", "salm2map_ms": e0.elapsed_time(e1), "map2salm_ms": e1.elapsed_time(e2),
                      "max_rel_error": rt_err,
                      "note": "separable: scrib200_theta_synth + phi-DFT GEMM, phi-DFT GEMM + scrib200_theta_quad; grid written to and read from HBM once"}
        del grid, back
        line = {
            "metric": "mode-timesteps/sec through ModesTimeSeries.grid_multiply (ell_max=32)", "value": float(n) * N / (ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"configs[3]: product of two ell<=32 mode series (spins 2 and -2) on the 129x129 working grid, output ell<=32, {N} time steps sharded by time",
                       "n_times": N, "n_modes": n, "grid": "129x129 (never formed in HBM)",
                       "l2": "explicit 256 MiB L2 flush between timed iterations; inputs + output 5.2 GB"},
            "roofline": {"kernel": "modes_product_kernel", "bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": dgemm, "unit": "TFLOP/s",
                         "frac": flops / (ms * 1e-3) / 1e12 / dgemm, "traffic": None,
                         "peak_source": "cuBLAS DGEMM 6144^3 measured in this run (MEASURED_PEAKS.json has no FP64 entry)",
                         "algorithmic_flops_per_launch": flops,
                         "note": "separable algorithm: theta synthesis + m-convolution + theta quadrature; the dense grid chain would need 70x the flops"},
            "cpu_baseline": {"value": float(n) * ns / cpu_s, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": f"first {ns} time steps through oracle.abd_ref.grid_multiply (restated spinsfast), {cpu_s:.1f} s; max rel. deviation of the GPU result {err:.1e}"},
            "grid_round_trip": round_trip,
            "e2e": None, "gpu_launches": int(launches), "clocks": clocks,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_timeshard_workload(args):
    """BASELINE configs[1] as ONE series sharded by TIME over the ranks (strong scaling): parallel.sharded_transform -
    point-to-point halo exchange of the input modes (NCCL), local synthesis / splines / analysis, no other collective.
    Optional workload, not the default bench line; device-resident."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import scri_b200 as sb
    from scri_b200 import _lib, ops, parallel
    from scri_b200.plan import TransformPlan

    kw = transformation_kwargs()
    N = args.n_times
    w = make_workload(N)
    lo, hi = parallel.shard_range(N, rank, world)
    t_d = ops.to_device(np.ascontiguousarray(w.t[lo:hi]))
    a_d = ops.to_device(np.ascontiguousarray(w.data[lo:hi]))
    plan = TransformPlan(w.ell_min, w.ell_max, w.dataType, r_is_scaled_out=w.r_is_scaled_out, **kw)
    halo = parallel.transform_halo(plan, float(w.t[lo]), float(w.t[hi - 1]), float(np.diff(w.t).min()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        u, m = parallel.sharded_transform(plan, t_d, a_d)
    barrier()
    l0 = _lib.launch_count()
    total = 0.0
    for _ in range(args.steps):
        flush.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        u, m = parallel.sharded_transform(plan, t_d, a_d)
        e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    ms = total / args.steps
    tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    n_out = torch.tensor([u.shape[0]], dtype=torch.int64, device="cuda")
    dist.all_reduce(n_out)
    if rank == 0:
        emit({
            "metric": METRIC, "value": float(w.n_modes) * N / (float(tms[0]) * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": float(tms[0]), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"configs[1] as one series of {N} steps sharded by time: halo of {halo} input samples per boundary exchanged point-to-point, no other collective",
                       "n_times": N, "n_out": int(n_out[0]), "n_modes": int(w.n_modes), "halo": halo, "l2": "explicit 256 MiB L2 flush between timed iterations"},
            "e2e": None, "gpu_launches": int(launches), "clocks": None,
        })
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n-times", type=int, default=100_000)
    ap.add_argument("--cpu-sample", type=int, default=4000, help="time steps in the cpu_baseline sample")
    ap.add_argument("--ref-sample", type=int, default=10_000, help="time steps per step of --impl reference")
    ap.add_argument("--workload", default="transform", choices=["transform", "batch", "product", "timeshard"],
                    help="transform = configs[1] (the bench line); batch = configs[2]; product = configs[3] (ell<=32 mode products)")
    ap.add_argument("--batch", type=int, default=4096, help="waveforms in the batch workload (all ranks together)")
    ap.add_argument("--no-extras", action="store_true", help="headline line only: skip the configs[2] batch and the time-sharded run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output times and modes to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs:
        if args.impl != "ours" or args.workload != "transform":
            ap.error("--dump-outputs covers the default transform workload of --impl ours")
        os.makedirs(args.dump_outputs, exist_ok=True)
    claim_stdout()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "batch":
        run_batch_workload(args)
    elif args.workload == "product":
        run_product_workload(args)
    elif args.workload == "timeshard":
        run_timeshard_workload(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
