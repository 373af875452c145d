"""Multi-GPU sharding of the transformation path (one process per GPU, torch.distributed).

The path shards two ways (SURVEY.md 8e):

* by waveform index - fully independent units, no data-path collective; `shard_range` gives each rank a
  contiguous slice of the batch and `gather_batch` is the optional final all_gather;
* by time - pointwise stages need nothing; the spline stages couple neighbouring samples only through the
  tridiagonal inverse, which decays like 0.268^k, so each rank takes its block plus a HALO-sample halo of
  *input modes* (`time_shard_with_halo`), transforms locally and keeps the outputs that fall in its own
  block (`owned_output_mask`).  The halo rows come from the neighbours by point-to-point exchange
  (`exchange_halos`) - 2 * HALO * n_modes * 16 bytes per boundary - and the results are all_gathered.

The host logic here is backend-agnostic: NCCL on GPUs, gloo in the CPU tests.
"""
import math

import numpy as np

HALO = 64


def shard_range(n_items, rank, world_size):
    """Contiguous [lo, hi) slice of `n_items` owned by `rank`; sizes differ by at most one."""
    base, extra = divmod(n_items, world_size)
    lo = rank * base + min(rank, extra)
    hi = lo + base + (1 if rank < extra else 0)
    return lo, hi


def time_shard_with_halo(n_times, rank, world_size, halo=HALO):
    """(lo, hi, lo_h, hi_h): owned block [lo, hi) and the block with halos [lo_h, hi_h)."""
    lo, hi = shard_range(n_times, rank, world_size)
    return lo, hi, max(0, lo - halo), min(n_times, hi + halo)


def owned_output_mask(uprm, t_global_first_owned, t_global_first_next, gamma, time_translation, is_last):
    """Outputs u'_i = (t_i - dt)/gamma belong to the rank that owns input sample i."""
    u_lo = (1 / gamma) * (t_global_first_owned - time_translation)
    if is_last:
        return uprm >= u_lo
    u_hi = (1 / gamma) * (t_global_first_next - time_translation)
    return (uprm >= u_lo) & (uprm < u_hi)


def exchange_halos(local, halo, group=None):
    """Send the first/last `halo` rows of `local` ([n_local, ...] tensor) to the previous/next rank.

    Returns (from_prev, from_next); None at the ends of the chain.  Works with NCCL (CUDA tensors) and gloo.
    """
    import torch
    import torch.distributed as dist

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    h = min(halo, local.shape[0])
    cplx = local.is_complex()
    wire = torch.view_as_real(local) if cplx else local                      # NCCL has no complex types
    staged = dist.get_backend(group) == "gloo" and wire.is_cuda             # gloo moves host memory
    dev = wire.device
    if staged:
        wire = wire[:h].cpu(), wire[-h:].cpu()
    else:
        wire = wire[:h].contiguous(), wire[-h:].contiguous()
    shape = (h,) + tuple(wire[0].shape[1:])
    from_prev = torch.empty(shape, dtype=wire[0].dtype, device=wire[0].device) if rank > 0 else None
    from_next = torch.empty(shape, dtype=wire[0].dtype, device=wire[0].device) if rank < world - 1 else None
    ops = []
    if rank > 0:
        ops.append(dist.P2POp(dist.isend, wire[0], rank - 1, group))
        ops.append(dist.P2POp(dist.irecv, from_prev, rank - 1, group))
    if rank < world - 1:
        ops.append(dist.P2POp(dist.isend, wire[1], rank + 1, group))
        ops.append(dist.P2POp(dist.irecv, from_next, rank + 1, group))
    if ops:
        for req in dist.batch_isend_irecv(ops):
            req.wait()

    def back(x):
        if x is None:
            return None
        if staged:
            x = x.to(dev)
        return torch.view_as_complex(x) if cplx else x

    return back(from_prev), back(from_next)


def gather_batch(local, counts, group=None):
    """all_gather of per-rank row blocks of unequal length `counts` (rows along dim 0)."""
    import torch
    import torch.distributed as dist

    world = dist.get_world_size(group)
    nmax = max(counts)
    pad = torch.zeros((nmax,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    if pad.is_complex():
        buf = torch.view_as_real(pad).contiguous()
        outs = [torch.empty_like(buf) for _ in range(world)]
        dist.all_gather(outs, buf, group=group)
        outs = [torch.view_as_complex(o) for o in outs]
    else:
        outs = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(outs, pad, group=group)
    return torch.cat([o[:c] for o, c in zip(outs, counts)], dim=0)


def sharded_time_derivative(t_local, data_local, order=1, halo=HALO, group=None):
    """d/dt (order 1 or 2) of a mode series sharded by TIME: every rank holds a contiguous block (ranks in time order).

    The cubic spline couples samples only through the tridiagonal inverse (0.268^k on uniform samples), so each rank
    borrows `halo` samples of t and of the modes from each neighbour (point-to-point, 2 * halo * (n_modes * 16 + 8) bytes
    per boundary - the only communication), differentiates its extended block on its own GPU (scrib200_spline_calculus)
    and keeps its own rows.  Replaces CubicSpline(t, data).derivative(order)(t) (scri/waveform_base.py:689-695) at scale."""
    import torch

    from . import ops

    prev_d, next_d = exchange_halos(data_local, halo, group)
    prev_t, next_t = exchange_halos(t_local, halo, group)
    parts_t = [x for x in (prev_t, t_local, next_t) if x is not None]
    parts_d = [x for x in (prev_d, data_local, next_d) if x is not None]
    ext = ops.spline_calculus(torch.cat(parts_t), torch.cat(parts_d), "derivative", order)
    lo = 0 if prev_t is None else prev_t.shape[0]
    return ext[lo : lo + t_local.shape[0]]


def sharded_fluxes(t_local, data_local, ell_min, ell_max, halo=HALO, group=None):
    """(energy, momentum, angular-momentum) fluxes of a strain series sharded by time (BASELINE config 5 across GPUs):
    one halo exchange for the time derivative, then every stage is pointwise in time.  Returns this rank's rows."""
    import math

    import torch

    from . import flux, ops

    hdot = sharded_time_derivative(t_local, data_local, 1, halo, group)
    edot = ops.norm(hdot) / (16.0 * math.pi)
    ev = ops.sparse_expectation(hdot, hdot, [flux.p_plus(ell_min, ell_max, s=-2), flux.p_minus(ell_min, ell_max, s=-2), flux.p_z(ell_min, ell_max, s=-2)])
    pdot = torch.stack([0.5 * (ev[:, 0].real + ev[:, 1].real), 0.5 * (ev[:, 0].imag - ev[:, 1].imag), ev[:, 2].real], dim=1) / (16.0 * math.pi)
    ev = ops.sparse_expectation(hdot, data_local, [flux.j_plus(ell_min, ell_max), flux.j_minus(ell_min, ell_max), flux.j_z(ell_min, ell_max)])
    jdot = torch.stack([0.5 * (ev[:, 0].real + ev[:, 1].real), 0.5 * (ev[:, 0].imag - ev[:, 1].imag), ev[:, 2].real], dim=1) / (-16.0 * math.pi)
    return edot, pdot, jdot


def transform_batch(plan, t, data_batch, companions=None):
    """Run one TransformPlan over a local shard `data_batch[B_local, N, n]` (device tensors): (u', modes'[B_local, N', n']).
    psi0..psi3 take their companion fields as [B_local, N, n_q] device tensors ordered psi(n+1)..psi4 (plan.run_batch)."""
    return plan.run_batch(t, data_batch, companions=companions)


def transform_batch_host(plan, t, data_host, sub_batch=None, out=None, companions_host=None):
    """BASELINE configs[2] from host memory: `data_host` [B, N, n_modes] complex128 numpy (this rank's shard of the batch;
    page-locked memory goes up by DMA, anything else through the staging ring) -> (u' [N'] numpy, modes' [B, N', n_out]
    numpy in pinned memory).  Sub-batches are double-buffered on the device: the H2D of sub-batch i+1 and the D2H of
    sub-batch i-1 run on their own streams under the kernels of sub-batch i (plan.run_batch).  `data_host` may also be a
    sequence of such arrays (a shard that lives in several host blocks): they flow through ONE pipeline without draining
    in between, and `out`, if given, is the matching sequence of result arrays (a list of results is returned).

    psi0..psi3 need `companions_host`, parallel to `data_host`: for one array, the sequence of Q host arrays
    [B, N, n_q] ordered psi(n+1)..psi4; for a sequence of blocks, one such sequence per block.  They go up with the
    sub-batch they belong to, in the same double-buffered pipeline.

    `sub_batch` defaults to 512 waveforms, and to 512 // (Q + 1) for a plan that mixes in Q companions, so that a psi plan
    needs no more device memory than an h plan.  Per waveform of N samples on G grid points, with n_q modes per field
    (16-byte complex), an h plan holds two input buffers (2 * 16 N n), the synthesized and the remapped grid (2 * 16 N G)
    and the modes (16 N' n_out); a psi plan holds 2 * 16 N sum(n_q) of inputs and, while it mixes, Q + 1 grids - on
    (Q + 1) times fewer waveforms.  At the shape of configs[2] (N = 2048, ell <= 8, G = 625) an h sub-batch of 512 holds
    2.6 GB of inputs and 21.0 GB of grids; a psi2 sub-batch of 170 (Q = 2) holds 2.7 GB of inputs and at most 10.4 GB of
    grids."""
    import ctypes

    import torch

    from . import _lib, ops

    single = isinstance(data_host, np.ndarray)
    blocks = [data_host] if single else list(data_host)
    n_comp = len(plan.mix)
    if n_comp and companions_host is None:
        raise ValueError("transform_batch_host of psi0..psi3 needs companions_host (host arrays of psi(n+1)..psi4)")
    if companions_host is not None and not n_comp:
        plan._check_companions(companions_host, (), host=True)   # raises: this plan mixes in no companion fields
    comp_blocks = [[]] * len(blocks)
    if n_comp:
        comp_blocks = [companions_host] if single else list(companions_host)
        if len(comp_blocks) != len(blocks):
            raise ValueError(f"companions_host has {len(comp_blocks)} blocks for {len(blocks)} blocks of data")
        comp_blocks = [plan._check_companions(cb, block.shape[:2], host=True) for block, cb in zip(blocks, comp_blocks)]
    outs = [out] if single else (list(out) if out is not None else [None] * len(blocks))
    blocks = [b if (b.dtype == np.complex128 and b.flags.c_contiguous) else np.ascontiguousarray(b, dtype=np.complex128) for b in blocks]
    N, n = blocks[0].shape[1:]
    if sub_batch is None:
        sub_batch = 512 // (n_comp + 1)
    sub = max(1, min(int(sub_batch), max(b.shape[0] for b in blocks)))
    lib = _lib.load()
    t_d = ops.to_device(t, np.float64)
    cur = torch.cuda.current_stream()
    cin, cout = torch.cuda.Stream(), torch.cuda.Stream()
    prep = plan.prepare(t_d)             # one time axis for the whole batch: its spline tables and retained block, once
    prep.resolve()
    bufs = [torch.empty((sub, N, n), dtype=torch.complex128, device="cuda") for _ in range(2)]
    cbufs = [[torch.empty((sub, N, mx["n_modes"]), dtype=torch.complex128, device="cuda") for mx in plan.mix] for _ in range(2)]
    free = [None, None]                                   # event: the kernels that read buffer b are done
    row_bytes = N * n * 16
    u_host = None
    i = 0
    for k, block in enumerate(blocks):
        B = block.shape[0]
        for b0 in range(0, B, sub):
            nb = min(sub, B - b0)
            b = i & 1
            i += 1
            if free[b] is not None:
                cin.wait_event(free[b])
            else:
                cin.wait_stream(cur)
            _lib.check(lib.scrib200_h2d(bufs[b].data_ptr(), block.ctypes.data + b0 * row_bytes, nb * row_bytes,
                                        ctypes.c_void_p(cin.cuda_stream)), "h2d")
            for c, cbuf in zip(comp_blocks[k], cbufs[b]):
                c_row = N * c.shape[2] * 16
                _lib.check(lib.scrib200_h2d(cbuf.data_ptr(), c.ctypes.data + b0 * c_row, nb * c_row, ctypes.c_void_p(cin.cuda_stream)),
                           "h2d")
            landed = torch.cuda.Event()
            landed.record(cin)
            cur.wait_event(landed)
            u, m = plan.run_batch(t_d, bufs[b][:nb], prep=prep, companions=[cb[:nb] for cb in cbufs[b]] if n_comp else None)
            done = torch.cuda.Event()
            done.record(cur)
            free[b] = done
            if outs[k] is None:
                outs[k] = torch.empty((B, m.shape[1], m.shape[2]), dtype=torch.complex128, pin_memory=True)
            elif not torch.is_tensor(outs[k]):
                outs[k] = torch.from_numpy(outs[k])
            cout.wait_event(done)
            with torch.cuda.stream(cout):
                outs[k][b0 : b0 + nb].copy_(m, non_blocking=True)
                if u_host is None:
                    u_host = torch.empty(u.shape, dtype=torch.float64, pin_memory=True)
                    u_host.copy_(u, non_blocking=True)
            m.record_stream(cout)
            u.record_stream(cout)
    cout.synchronize()
    cur.synchronize()
    results = [o.numpy() for o in outs]
    return u_host.numpy(), (results[0] if single else results)


SPLINE_DECAY_ROWS = 40   # rows after which a not-a-knot spline has forgotten its end conditions (0.268^40 ~ 1e-23)


def transform_halo(plan, t_first, t_last, dt_min):
    """Input samples a rank must borrow from each neighbour to transform its block of [t_first, t_last] alone.

    The output of input sample i sits at u'_i = (t_i - dt)/gamma; grid point g evaluates its spline there, i.e. at the
    input time t* with k_g (t* - alpha_g) = u'_i.  With 1/(gamma k_g) = 1 - v.r_g the distance is
    |t* - t_i| = |alpha_g - dt (1 - v.r_g) - t_i v.r_g|: bounded for supertranslations and rotations, growing like beta |t|
    under a boost.  Linear in t_i, so the block's ends give the maximum."""
    k = np.asarray(plan.kconformal, dtype=float)
    alpha = np.asarray(plan.alpha, dtype=float)
    one_minus_vr = 1.0 / (plan.gamma * k)
    drift = 0.0
    for ti in (t_first, t_last):
        drift = max(drift, float(np.abs(alpha - plan.time_translation * one_minus_vr - ti * (1.0 - one_minus_vr)).max()))
    return int(math.ceil(drift / dt_min)) + SPLINE_DECAY_ROWS + 2


def sharded_transform(plan, t_local, data_local, companions_local=None, halo=None, group=None, timings=None):
    """WaveformModes.transform (scri/waveform_grid.py:331-630) of ONE long series sharded by TIME: every rank holds a
    contiguous block of (t, modes), ranks in time order.  Each rank borrows `halo` input samples from its neighbours
    (point-to-point: the only data-path communication besides the few scalars below), synthesizes the extended block,
    builds the splines of the extended block and evaluates them at the output times of the samples it owns, masked by the
    GLOBAL retained range; the analysis is pointwise in time.  Returns (u'_local, modes'_local); `gather_batch` assembles
    the full series where wanted.  `halo=None` sizes the halo from the transformation (`transform_halo`); a boost needs
    beta |t| / dt extra samples, and when that exceeds a neighbour's block the call refuses (shard by waveform instead).

    psi0..psi3 need `companions_local`: this rank's block of each higher Weyl scalar, [n_local, n_q] device tensors ordered
    psi(n+1)..psi4.  The same halo is borrowed for each of them, and the extended block is synthesized and mixed with the
    extended time axis.  The mixing is pointwise in time and the spline acts on the mixed grid, so the halo does not grow."""
    import torch
    import torch.distributed as dist

    if plan.mix and companions_local is None:
        raise ValueError("sharded_transform of psi0..psi3 needs companions_local=[psi(n+1), ..., psi4] as device tensors")
    plan._check_companions(companions_local, (int(data_local.shape[0]),))
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    dev = t_local.device
    n_loc = int(t_local.shape[0])
    step = (t_local[1:] - t_local[:-1]).min() if n_loc > 1 else torch.tensor(float("inf"), dtype=torch.float64, device=dev)
    mine = torch.stack([t_local[0], t_local[-1], step, torch.tensor(float(n_loc), dtype=torch.float64, device=dev)])
    wire = mine.cpu() if dist.get_backend(group) == "gloo" else mine
    ends = [torch.empty_like(wire) for _ in range(world)]

    def mark(name):                                                          # `timings`: name -> CUDA timing event
        if timings is not None and dev.type == "cuda":
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            timings[name] = ev

    mark("all_gather_begin")
    dist.all_gather(ends, wire, group=group)
    mark("all_gather_end")
    ends = torch.stack(ends).cpu().numpy()                                   # [world, 4]: first, last, min step, samples
    t0, tN = float(ends[0, 0]), float(ends[-1, 1])
    gaps = ends[1:, 0] - ends[:-1, 1]
    dt_min = float(min(ends[:, 2].min(), gaps.min() if gaps.size else np.inf))
    if halo is None:
        halo = max(transform_halo(plan, float(ends[r, 0]), float(ends[r, 1]), dt_min) for r in range(world))
    if world > 1 and halo > int(ends[:, 3].min()):
        raise ValueError(
            f"time-sharded transform needs a halo of {halo} input samples but the smallest block has {int(ends[:, 3].min())}: "
            "the boost moves the input window of late output times too far; shard by waveform index instead"
        )
    mark("halo_begin")
    prev_d, next_d = exchange_halos(data_local, halo, group)
    prev_t, next_t = exchange_halos(t_local, halo, group)
    c_ext = None
    if companions_local is not None:
        c_ext = []
        for c in companions_local:
            prev_c, next_c = exchange_halos(c, halo, group)
            c_ext.append(torch.cat([x for x in (prev_c, c, next_c) if x is not None]))
    mark("halo_end")
    t_ext = torch.cat([x for x in (prev_t, t_local, next_t) if x is not None])
    d_ext = torch.cat([x for x in (prev_d, data_local, next_d) if x is not None])
    F = plan.synthesize(d_ext, t_ext, companions=c_ext)
    prep = plan.prepare(t_ext)                                              # spline factor table of the extended block
    # output times of the samples this rank owns, masked by the global retained range (waveform_grid.py:564-568)
    if plan.divide_by_gamma:
        u_all = (t_local - plan.time_translation) / plan.gamma
    else:
        u_all = (1 / plan.gamma) * (t_local - plan.time_translation)
    u_min = (plan.d_k * (t0 - plan.d_alpha)).max()
    u_max = (plan.d_k * (tN - plan.d_alpha)).min()
    uprm = u_all[(u_all >= u_min) & (u_all <= u_max)].contiguous()
    n_out = int(uprm.shape[0])
    if n_out == 0:
        return uprm, torch.empty((0, plan.n_modes_out), dtype=torch.complex128, device=dev)
    torch.cuda.current_stream().wait_event(prep.done)
    return uprm, plan.remap_analyze(t_ext, F, uprm, prep, plan.analysis)
