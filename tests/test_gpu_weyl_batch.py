"""Weyl scalars psi0..psi3 in the batched, graph-captured and time-sharded transforms.

Under a BMS transformation psi_n picks up the higher Weyl scalars psi_{n+1}..psi4 times powers of a factor that depends on
time and grid point (scri/waveform_grid.py:504-550), so each of these paths takes the companion fields per call
(`companions=`) and mixes them with scrib200_weyl_mix_series (mix.cu).  The single-waveform transform of psi0..psi3 is
pinned against the reference's output and the oracle elsewhere; here it is the exact oracle of the new paths:
  * run_batch equals per-waveform run bit for bit, one waveform is within 1e-12 of the oracle, transform_batch_host
    (pinned and pageable companions) equals run_batch bit for bit, and the reference fixtures full_psi3 / full_psi2 go
    through run_batch;
  * scrib200_weyl_mix_series through the C ABI: poisoned outputs with guard rows, per-series scrib200_weyl_mix bit for bit,
    sampled elements within gamma S of a long-double Horner evaluation (kernel_check.py), row counts past the 65535-CTA
    grid limit of scrib200_weyl_mix;
  * a captured graph replays run(..., companions=...) and follows new contents of the companion tensors;
  * a time-sharded psi2 over two gloo ranks against the single-process transform;
  * malformed companions raise ValueError before any launch."""
import ctypes
import os

import numpy as np
import pytest

import scri_b200 as sb
from kernel_check import GUARD, _note, _poisoned, _torch, check_close, check_guard
from oracle import scri_ref as R
from scri_b200 import _lib, ops, parallel
from scri_b200 import plan as P
from scri_inputs import real_supertranslation, smooth_modes

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-12        # BASELINE.json north_star: 1e-12 relative (FP64)
BMS = dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03])
WEYL = [sb.psi0, sb.psi1, sb.psi2, sb.psi3]


def rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def wm(t, data, ell_min, dataType, ell_max=8):
    return sb.WaveformModes(t=t.copy(), data=data.copy(), ell_min=ell_min, ell_max=ell_max, frameType=sb.Inertial, dataType=dataType,
                            r_is_scaled_out=True, m_is_scaled_out=True)


def key(DT):
    return "psi{}_modes".format(sb.DataNames[DT][-1])


def weyl_batch(dataType, B, N, t0=0.0, t1=60.0, seed=0):
    """t [N] and, for every Weyl scalar DT = dataType..psi4, modes [B, N, n_DT] with ell from |s_DT| to 8."""
    fields = {}
    for DT in range(dataType, sb.psi4 + 1):
        s = abs(sb.SpinWeights[DT])
        fields[DT] = np.stack([smooth_modes(n_times=N, ell_min=s, t0=t0, t1=t1, seed=seed + 100 * DT + b)[1] for b in range(B)])
    t = np.linspace(t0, t1, N)
    return t, fields


def weyl_plan(dataType, t, fields, b=0, **kw):
    """TransformPlan of `dataType` whose bound companions are waveform b of the batch."""
    extra = {key(DT): wm(t, fields[DT][b], abs(sb.SpinWeights[DT]), DT) for DT in range(dataType + 1, sb.psi4 + 1)}
    return P.TransformPlan(abs(sb.SpinWeights[dataType]), 8, dataType, r_is_scaled_out=True, **kw, **extra)


# ------------------------------------------------------------------------------------------------------------ batch
@pytest.mark.parametrize("dataType", WEYL, ids=["psi0", "psi1", "psi2", "psi3"])
def test_run_batch_equals_single_runs_and_the_oracle(dataType):
    """psi0..psi3 with 4..1 companions (psi0 reaches the kernel's five fields): run_batch against per-waveform run with the
    same companions (bit for bit), the bound companions (bit for bit for waveform 0), the oracle (1e-12), transform_batch
    and transform_batch_host with pageable and page-locked companions (bit for bit)."""
    torch = _torch()
    B, N = 5, 333
    t, f = weyl_batch(dataType, B, N)
    pl = weyl_plan(dataType, t, f, **BMS)
    assert len(pl.mix) == sb.psi4 - dataType
    td, bd = ops.to_device(t), ops.to_device(f[dataType])
    comps = [ops.to_device(f[DT]) for DT in range(dataType + 1, sb.psi4 + 1)]
    up, out = pl.run_batch(td, bd, companions=comps)
    assert out.shape == (B, up.shape[0], pl.n_modes_out)
    for b in range(B):
        up1, out1 = pl.run(td, bd[b].contiguous(), companions=[c[b].contiguous() for c in comps])
        assert torch.equal(up1, up) and torch.equal(out1, out[b]), b
    up0, out0 = pl.run(td, bd[0].contiguous())                       # the companions bound when the plan was built
    assert torch.equal(up0, up) and torch.equal(out0, out[0])
    b = 3
    ref = R.transform(R.Modes(t=t, data=f[dataType][b].copy(), ell_min=abs(sb.SpinWeights[dataType]), dataType=dataType), **BMS,
                      **{key(DT): R.Modes(t=t, data=f[DT][b].copy(), ell_min=abs(sb.SpinWeights[DT]), dataType=DT)
                         for DT in range(dataType + 1, sb.psi4 + 1)})
    assert np.array_equal(up.cpu().numpy(), ref.t)
    assert rel(out[b].cpu().numpy(), ref.data) < RTOL
    up2, out2 = parallel.transform_batch(pl, td, bd, companions=comps)
    assert torch.equal(up2, up) and torch.equal(out2, out)
    pageable = [f[DT] for DT in range(dataType + 1, sb.psi4 + 1)]
    pinned = []
    for c in pageable:
        p = torch.empty(c.shape, dtype=torch.complex128, pin_memory=True)
        p.numpy()[...] = c
        pinned.append(p.numpy())
    for host in (pageable, pinned):
        uh, mh = parallel.transform_batch_host(pl, t, f[dataType], sub_batch=2, companions_host=host)
        assert np.array_equal(uh, up.cpu().numpy()) and np.array_equal(mh, out.cpu().numpy())


def test_transform_batch_host_blocks_and_default_sub_batch():
    """Several host blocks, each with its own companions, through one pipeline; and the default sub-batch."""
    B, N = 4, 257
    t, f = weyl_batch(sb.psi2, B, N, seed=7)
    pl = weyl_plan(sb.psi2, t, f, **BMS)
    comps = [ops.to_device(f[DT]) for DT in (sb.psi3, sb.psi4)]
    up, out = pl.run_batch(ops.to_device(t), ops.to_device(f[sb.psi2]), companions=comps)
    cuts = [(0, 1), (1, 4)]
    uh, res = parallel.transform_batch_host(pl, t, [f[sb.psi2][lo:hi] for lo, hi in cuts], sub_batch=2,
                                            companions_host=[[f[sb.psi3][lo:hi], f[sb.psi4][lo:hi]] for lo, hi in cuts])
    assert np.array_equal(uh, up.cpu().numpy())
    assert np.array_equal(np.concatenate(res), out.cpu().numpy())
    uh, mh = parallel.transform_batch_host(pl, t, f[sb.psi2], companions_host=[f[sb.psi3], f[sb.psi4]])   # 170: one sub-batch
    assert np.array_equal(mh, out.cpu().numpy())


def test_reference_fixtures_through_run_batch():
    """The reference's own output for psi3 (with psi4) and psi2 (with psi3, psi4) under the full transformation, through
    run_batch with one waveform and with the waveform repeated three times: u' bit-exact, modes within 1e-12, and the
    repeated rows equal to the single one bit for bit."""
    torch = _torch()
    g = np.load(os.path.join(GOLD, "reference_transform.npz"))
    kw = dict(supertranslation=g["supertranslation"], frame_rotation=g["frame_rotation"], boost_velocity=g["boost_velocity"])
    t = g["psi_t"]
    w = {sb.psi4: wm(t, g["psi4_in"], 2, sb.psi4), sb.psi3: wm(t, g["psi3_in"], 1, sb.psi3), sb.psi2: wm(t, g["psi2_in"], 0, sb.psi2)}
    td = ops.to_device(t)
    for dataType, name in ((sb.psi3, "full_psi3"), (sb.psi2, "full_psi2")):
        pl = P.TransformPlan(w[dataType].ell_min, w[dataType].ell_max, dataType, r_is_scaled_out=True,
                             **{key(DT): w[DT] for DT in range(dataType + 1, sb.psi4 + 1)}, **{k: np.copy(v) for k, v in kw.items()})
        d = ops.to_device(w[dataType].data)
        comps = [ops.to_device(w[DT].data) for DT in range(dataType + 1, sb.psi4 + 1)]
        u1, m1 = pl.run_batch(td, d[None].contiguous(), companions=[c[None].contiguous() for c in comps])
        assert np.array_equal(u1.cpu().numpy(), g[f"{name}_t"]), name
        assert rel(m1[0].cpu().numpy(), g[f"{name}_data"]) < RTOL, name
        u3, m3 = pl.run_batch(td, d[None].repeat(3, 1, 1), companions=[c[None].repeat(3, 1, 1) for c in comps])
        assert torch.equal(u3, u1)
        for b in range(3):
            assert torch.equal(m3[b], m1[0]), (name, b)


# ------------------------------------------------------------------------------------------------------------ kernel
def _mix_reference(Fs, coefs, t_rows, alpha, A, C, scale, off):
    """out = scale (sum_q c_q F_q z^q - off), z = (t - alpha) A - C, by Horner's rule in long double; and S, the same over
    absolute values with |z| replaced by |A||t - alpha| + |C| (|x| = |Re x| + |Im x|): what bounds the rounding of z."""
    ld, cld = np.longdouble, np.clongdouble
    absc = lambda x: np.abs(x.real) + np.abs(x.imag)
    dt = t_rows[:, None].astype(ld) - alpha[None, :].astype(ld)
    z = dt * A[None, :].astype(cld) - C[None, :].astype(cld)
    Z = absc(A)[None, :] * np.abs(dt.astype(float)) + absc(C)[None, :]
    nq = len(Fs)
    acc = ld(coefs[-1]) * Fs[-1].astype(cld)
    S = abs(coefs[-1]) * absc(Fs[-1])
    for q in range(nq - 2, -1, -1):
        acc = acc * z + ld(coefs[q]) * Fs[q].astype(cld)
        S = S * Z + abs(coefs[q]) * absc(Fs[q])
    ref = scale[None, :].astype(ld) * (acc - off[None, :].astype(cld))
    return ref, np.abs(scale)[None, :] * (S + absc(off)[None, :])


class MixCase:
    """Device buffers of one scrib200_weyl_mix_series case: fields [rows + GUARD, 2G] float64 (complex128 rows) with poisoned
    guard rows, t [n_times], the per-point tables, and helpers that launch either entry point into a poisoned output."""

    def __init__(self, n_fields, with_offset, G, n_times, n_series, seed):
        torch = _torch()
        self.nq, self.G, self.n_times, self.n_series = n_fields, G, n_times, n_series
        self.rows = n_times * n_series
        gen = torch.Generator(device="cuda").manual_seed(seed)
        rng = np.random.default_rng(seed)
        self.F = []
        for _ in range(n_fields):
            buf = _poisoned((self.rows + GUARD, 2 * G))
            buf[: self.rows] = torch.randn((self.rows, 2 * G), dtype=torch.float64, device="cuda", generator=gen)
            self.F.append(buf)
        self.coefs = [float(c) for c in rng.choice([1.0, 4.0, 6.0, 5.0, 10.0], size=n_fields)]
        self.coefs[0] = 1.0
        self.t_h = np.sort(rng.uniform(-50.0, 150.0, n_times))
        self.alpha_h = rng.uniform(-1.0, 1.0, G)
        self.A_h = 0.02 * (rng.normal(size=G) + 1j * rng.normal(size=G))
        self.C_h = 0.05 * (rng.normal(size=G) + 1j * rng.normal(size=G))
        self.scale_h = rng.uniform(0.5, 2.0, G)
        self.off_h = (rng.normal(size=G) + 1j * rng.normal(size=G)) if with_offset else np.zeros(G, dtype=complex)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.t, self.alpha, self.A, self.C, self.scale = dev(self.t_h), dev(self.alpha_h), dev(self.A_h), dev(self.C_h), dev(self.scale_h)
        self.off = dev(self.off_h) if with_offset else None

    def _args(self, field_ptrs):
        ptrs = (ctypes.c_void_p * self.nq)(*field_ptrs)
        return ptrs, (ctypes.c_double * self.nq)(*self.coefs)

    def series(self, out, alias=False):
        """One scrib200_weyl_mix_series launch over the whole batch into `out` (with `alias`, `out` is field 0)."""
        lib = _lib.load()
        ptrs, cf = self._args([out.data_ptr() if (alias and q == 0) else f.data_ptr() for q, f in enumerate(self.F)])
        _lib.check(lib.scrib200_weyl_mix_series(
            ptrs, cf, self.nq, _lib.ptr(self.t), self.n_times, self.n_series, self.G, _lib.ptr(self.alpha), _lib.ptr(self.A),
            _lib.ptr(self.C), _lib.ptr(self.scale), _lib.ptr(self.off) if self.off is not None else None, _lib.ptr(out),
            _lib.stream_ptr()), "weyl_mix_series")

    def single(self, out, row0, n_rows, t_ptr):
        """scrib200_weyl_mix over rows [row0, row0 + n_rows) of every field, reading t from `t_ptr`."""
        lib = _lib.load()
        off = row0 * self.G * 16
        ptrs, cf = self._args([f.data_ptr() + off for f in self.F])
        _lib.check(lib.scrib200_weyl_mix(
            ptrs, cf, self.nq, ctypes.c_void_p(t_ptr), n_rows, self.G, _lib.ptr(self.alpha), _lib.ptr(self.A), _lib.ptr(self.C),
            _lib.ptr(self.scale), _lib.ptr(self.off) if self.off is not None else None, ctypes.c_void_p(out.data_ptr() + off),
            _lib.stream_ptr()), "weyl_mix")

    def check_rows(self, out_host, rows, what):
        """Rows `rows` of the output against the long-double reference; returns max |out - ref| / (gamma S)."""
        Fs = [f[torch_index(rows)].cpu().numpy().view(complex) for f in self.F]
        ref, S = _mix_reference(Fs, self.coefs, self.t_h[rows % self.n_times], self.alpha_h, self.A_h, self.C_h, self.scale_h, self.off_h)
        return check_close(out_host[rows].view(complex), ref, S, 4 * self.nq + 4, what)


def torch_index(rows):
    return _torch().from_numpy(np.asarray(rows, dtype=np.int64)).cuda()


def _sample_rows(case, rng, every_row_below=6000):
    if case.rows <= every_row_below:
        return np.arange(case.rows)
    rows = set()
    for s in {0, 1, case.n_series // 2, case.n_series - 1}:
        for i in {0, 1, 63, 64, case.n_times // 2, case.n_times - 2, case.n_times - 1}:
            if 0 <= i < case.n_times:
                rows.add(s * case.n_times + i)
    rows.update(rng.integers(0, case.rows, 200).tolist())
    return np.array(sorted(r for r in rows if 0 <= r < case.rows))


def _run_series_checks(case, reference_out, what):
    """The batch into a poisoned buffer: guard intact, equal to `reference_out` (scrib200_weyl_mix) bit for bit, sampled
    rows within gamma S of long double; then in place (out = field 0): the same bits, the guard of field 0 intact."""
    torch = _torch()
    out = _poisoned((case.rows + GUARD, 2 * case.G))
    case.series(out)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    check_guard(o, case.rows, f"{what} output")
    r = reference_out.cpu().numpy()
    check_guard(r, case.rows, f"{what} weyl_mix output")
    assert np.array_equal(o[: case.rows].view(np.int64), r[: case.rows].view(np.int64)), f"{what}: differs from scrib200_weyl_mix"
    _note("weyl_mix_series_kernel", case.check_rows(o, _sample_rows(case, np.random.default_rng(case.rows)), what))
    inplace = case.F[0].clone()
    case.series(inplace, alias=True)
    torch.cuda.synchronize()
    ip = inplace.cpu().numpy()
    check_guard(ip, case.rows, f"{what} in place")
    assert np.array_equal(ip[: case.rows].view(np.int64), o[: case.rows].view(np.int64)), f"{what}: in place differs"


SMALL_SHAPES = {1: (200, 333), 2: (625, 100), 3: (129, 1), 4: (1, 64), 5: (333, 65)}   # n_fields -> (G, n_times)


@pytest.mark.parametrize("n_series", [1, 7])
@pytest.mark.parametrize("with_offset", [False, True], ids=["no-offset", "offset"])
@pytest.mark.parametrize("n_fields", [1, 2, 3, 4, 5])
def test_weyl_mix_series_kernel(n_fields, with_offset, n_series):
    """n_fields 1..5 with and without the offset, G and n_times around the 128-point CTA and the 64-row slab, one series
    and seven: equal to scrib200_weyl_mix run series by series, and to a long-double Horner evaluation."""
    torch = _torch()
    G, n_times = SMALL_SHAPES[n_fields]
    case = MixCase(n_fields, with_offset, G, n_times, n_series, seed=10 * n_fields + n_series + with_offset)
    ref = _poisoned((case.rows + GUARD, 2 * G))
    for s in range(n_series):
        case.single(ref, s * n_times, n_times, case.t.data_ptr())
    torch.cuda.synchronize()
    _run_series_checks(case, ref, f"weyl_mix_series nq={n_fields} offset={with_offset} G={G} N={n_times} x {n_series}")


def test_weyl_mix_series_past_the_grid_limit_of_weyl_mix():
    """Row counts scrib200_weyl_mix cannot launch (it puts ceil(rows / 64) CTAs in gridDim.y, at most 65535, i.e. 4.19 M
    rows): 2049 series of 2048 steps (4.2 M rows, against scrib200_weyl_mix series by series); one series of 4.2 M steps
    (the slabs stride over gridDim.y; against scrib200_weyl_mix on two halves); 70001 series of 3 steps (the series stride
    over gridDim.z; against one scrib200_weyl_mix launch on the time axis tiled 70001 times)."""
    torch = _torch()
    limit = 65535 * 64
    case = MixCase(3, True, 5, 2048, 2049, seed=1)
    assert case.rows > limit
    ref = _poisoned((case.rows + GUARD, 2 * case.G))
    for s in range(case.n_series):
        case.single(ref, s * case.n_times, case.n_times, case.t.data_ptr())
    torch.cuda.synchronize()
    _run_series_checks(case, ref, "2049 x 2048")
    del case, ref

    case = MixCase(2, False, 3, 4_200_000, 1, seed=2)
    assert case.rows > limit
    ref = _poisoned((case.rows + GUARD, 2 * case.G))
    half = case.rows // 2
    case.single(ref, 0, half, case.t.data_ptr())
    case.single(ref, half, case.rows - half, case.t.data_ptr() + 8 * half)
    torch.cuda.synchronize()
    _run_series_checks(case, ref, "1 x 4.2e6")
    del case, ref

    case = MixCase(2, True, 3, 3, 70_001, seed=3)
    tiled = case.t.repeat(case.n_series)
    ref = _poisoned((case.rows + GUARD, 2 * case.G))
    case.single(ref, 0, case.rows, tiled.data_ptr())
    torch.cuda.synchronize()
    _run_series_checks(case, ref, "70001 x 3")


def test_weyl_mix_series_argument_errors():
    torch = _torch()
    case = MixCase(2, False, 8, 10, 2, seed=4)
    out = _poisoned((case.rows + GUARD, 2 * case.G))
    lib = _lib.load()
    before = _lib.launch_count()
    for nq in (0, 6):
        ptrs = (ctypes.c_void_p * 6)(*([case.F[0].data_ptr()] * 6))
        cf = (ctypes.c_double * 6)(*([1.0] * 6))
        with pytest.raises(_lib.Scrib200Error, match="n_fields"):
            _lib.check(lib.scrib200_weyl_mix_series(ptrs, cf, nq, _lib.ptr(case.t), 10, 2, 8, _lib.ptr(case.alpha), _lib.ptr(case.A),
                                                    _lib.ptr(case.C), _lib.ptr(case.scale), None, _lib.ptr(out), _lib.stream_ptr()))
    ptrs = (ctypes.c_void_p * 2)(case.F[0].data_ptr(), case.F[1].data_ptr() + 8)
    cf = (ctypes.c_double * 2)(1.0, 1.0)
    with pytest.raises(_lib.Scrib200Error, match="misaligned"):
        _lib.check(lib.scrib200_weyl_mix_series(ptrs, cf, 2, _lib.ptr(case.t), 10, 2, 8, _lib.ptr(case.alpha), _lib.ptr(case.A),
                                                _lib.ptr(case.C), _lib.ptr(case.scale), None, _lib.ptr(out), _lib.stream_ptr()))
    ptrs = (ctypes.c_void_p * 2)(case.F[0].data_ptr(), case.F[1].data_ptr())
    _lib.check(lib.scrib200_weyl_mix_series(ptrs, cf, 2, _lib.ptr(case.t), 10, 0, 8, _lib.ptr(case.alpha), _lib.ptr(case.A),
                                            _lib.ptr(case.C), _lib.ptr(case.scale), None, _lib.ptr(out), _lib.stream_ptr()))
    assert _lib.launch_count() == before                  # nothing launched, and no series is no work
    torch.cuda.synchronize()
    check_guard(out.cpu().numpy(), 0, "untouched output")


# ------------------------------------------------------------------------------------------------------------ capture
def test_captured_psi2_replays_run_with_companions():
    """TransformPlan.capture of psi2: the replay equals run(..., companions=...) bit for bit; after new values are written
    into the captured companion tensors in place, the next replay equals a fresh run on them."""
    torch = _torch()
    t, f = weyl_batch(sb.psi2, 1, 4000, t0=0.0, t1=400.0, seed=11)
    pl = weyl_plan(sb.psi2, t, f, **BMS)
    td, ad = ops.to_device(t), ops.to_device(f[sb.psi2][0])
    comps = [ops.to_device(f[DT][0]) for DT in (sb.psi3, sb.psi4)]
    u1, m1 = pl.run(td, ad, companions=comps)
    cap = pl.capture(td, ad, companions=comps)
    u2, m2 = cap.replay()
    assert cap.verify()
    assert torch.equal(u1, u2) and torch.equal(m1, m2)
    comps[0].mul_(-0.5 + 0.25j)
    comps[1].copy_(comps[1].flip(1))
    u3, m3 = cap.replay()
    torch.cuda.synchronize()
    u4, m4 = pl.run(td, ad, companions=comps)
    assert torch.equal(u3, u4) and torch.equal(m3, m4)
    assert not torch.equal(m3, m1)


# ------------------------------------------------------------------------------------------------------------ time shard
def _sharded_psi2_worker(rank, world, port, q, kw, n_times, t1):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        t, f = weyl_batch(sb.psi2, 1, n_times, t0=0.0, t1=t1, seed=29)
        lo, hi = parallel.shard_range(t.size, rank, world)
        tl = t[lo:hi].copy()
        local = {DT: f[DT][0, lo:hi].copy() for DT in f}
        plan = P.TransformPlan(0, 8, sb.psi2, r_is_scaled_out=True, **kw,
                               **{key(DT): wm(tl, local[DT], abs(sb.SpinWeights[DT]), DT) for DT in (sb.psi3, sb.psi4)})
        try:
            u, m = parallel.sharded_transform(plan, ops.to_device(tl), ops.to_device(local[sb.psi2]),
                                              [ops.to_device(local[DT]) for DT in (sb.psi3, sb.psi4)])
            q.put((rank, u.cpu().numpy(), m.cpu().numpy(), None))
        except ValueError as e:
            q.put((rank, None, None, str(e)))
    finally:
        dist.destroy_process_group()


def _run_sharded(kw, n_times, t1, world=2):
    import socket

    import torch.multiprocessing as mp

    s_ = socket.socket()
    s_.bind(("127.0.0.1", 0))
    port = s_.getsockname()[1]
    s_.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_psi2_worker, args=(r, world, port, q, kw, n_times, t1)) for r in range(world)]
    for pr in procs:
        pr.start()
    res = sorted([q.get(timeout=300) for _ in range(world)], key=lambda x: x[0])
    for pr in procs:
        pr.join(timeout=60)
    return res


def test_time_sharded_psi2_world2():
    """psi2 with psi3 and psi4 sharded by time over two gloo ranks, under supertranslation + rotation + boost over 4000
    steps of 100 M: u' bit-exact and modes within 1e-12 of the single-process w.transform(psi3_modes=, psi4_modes=).  A
    boost that needs more than a block of halo is still refused with the same message."""
    kw = dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03])
    res = _run_sharded(kw, 4000, 100.0)
    assert all(r[3] is None for r in res), res[0][3]
    t, f = weyl_batch(sb.psi2, 1, 4000, t0=0.0, t1=100.0, seed=29)
    ref = wm(t, f[sb.psi2][0], 0, sb.psi2).transform(psi3_modes=wm(t, f[sb.psi3][0], 1, sb.psi3),
                                                      psi4_modes=wm(t, f[sb.psi4][0], 2, sb.psi4), **kw)
    u = np.concatenate([r[1] for r in res])
    m = np.concatenate([r[2] for r in res])
    assert np.array_equal(u, ref.t)
    assert rel(m, ref.data) < RTOL
    res = _run_sharded(dict(boost_velocity=[0.3, 0.4, 0.5]), 4000, 400.0)
    assert all(r[3] is not None and "shard by waveform" in r[3] for r in res)


# ------------------------------------------------------------------------------------------------------------ errors
def test_malformed_companions_raise_before_any_launch():
    """Wrong count, order, shape, dtype, device, contiguity or row count, companions given to a plan without mixing, and
    psi paths that cannot use the bound fields called without companions: ValueError, and no kernel launched."""
    torch = _torch()
    B, N = 2, 120
    t, f = weyl_batch(sb.psi2, B, N, seed=5)
    pl = weyl_plan(sb.psi2, t, f, **BMS)
    td, bd = ops.to_device(t), ops.to_device(f[sb.psi2])
    c3, c4 = ops.to_device(f[sb.psi3]), ops.to_device(f[sb.psi4])
    h = P.TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **BMS)
    hd = ops.to_device(np.stack([smooth_modes(n_times=N, t0=0.0, t1=60.0, seed=b)[1] for b in range(B)]))
    assert c3.shape[-1] != c4.shape[-1]                   # ell from 1 and from 2: a swapped order shows in the shapes
    batch_cases = {
        "one field": [c3],
        "three fields": [c3, c4, c4],
        "swapped": [c4, c3],
        "a stacked tensor": torch.stack([c3[..., :77], c4]),
        "rows": [c3[:, :-1].contiguous(), c4[:, :-1].contiguous()],
        "batch": [c3[:1].contiguous(), c4[:1].contiguous()],
        "complex64": [c3.to(torch.complex64), c4],
        "float64": [torch.view_as_real(c3)[..., 0].contiguous(), c4],
        "host": [f[sb.psi3], f[sb.psi4]],
        "cpu tensor": [c3.cpu(), c4],
        "not contiguous": [c3.transpose(0, 1).contiguous().transpose(0, 1), c4],
        "missing": None,
    }
    before = _lib.launch_count()
    for what, comps in batch_cases.items():
        with pytest.raises(ValueError):
            pl.run_batch(td, bd, companions=comps)
        with pytest.raises(ValueError):
            parallel.transform_batch(pl, td, bd, companions=comps)
        if isinstance(comps, list) and what != "batch":          # the same fields, one waveform's worth, for run / synthesize / capture
            single = [c[0] if torch.is_tensor(c) else c for c in comps]
            for call in (lambda: pl.run(td, bd[0], companions=single), lambda: pl.synthesize(bd[0], td, companions=single),
                         lambda: pl.capture(td, bd[0], companions=single)):
                with pytest.raises(ValueError):
                    call()
    with pytest.raises(ValueError):
        pl.capture(td, bd[0])
    host_cases = {"missing": None, "one field": [f[sb.psi3]], "swapped": [f[sb.psi4], f[sb.psi3]],
                  "rows": [f[sb.psi3][:, 1:], f[sb.psi4][:, 1:]], "device": [c3, c4]}
    for what, comps in host_cases.items():
        with pytest.raises(ValueError):
            parallel.transform_batch_host(pl, t, f[sb.psi2], companions_host=comps)
    with pytest.raises(ValueError):
        parallel.transform_batch_host(pl, t, [f[sb.psi2]], companions_host=[[f[sb.psi3], f[sb.psi4]], [f[sb.psi3], f[sb.psi4]]])
    for call in (lambda: h.run_batch(td, hd, companions=[c3]), lambda: h.run(td, hd[0], companions=[c3[0]]),
                 lambda: h.synthesize(hd[0], td, companions=[c3[0]]), lambda: h.capture(td, hd[0], companions=[c3[0]]),
                 lambda: parallel.transform_batch_host(h, t, hd.cpu().numpy(), companions_host=[f[sb.psi3]]),
                 lambda: parallel.sharded_transform(h, td, hd[0], [c3[0]]),
                 lambda: parallel.sharded_transform(pl, td, bd[0])):
        with pytest.raises(ValueError):
            call()
    assert _lib.launch_count() == before
