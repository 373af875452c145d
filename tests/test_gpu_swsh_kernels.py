"""Every launch branch of the SWSH synthesis (synth.cu), the device-built synthesis table (mix.cu:swsh_pack) and the SWSH
analysis (analysis.cu) against a plain high-precision reference of the same operation, through the C ABI.

Each case allocates its own buffers so that it can poison them: outputs start as NaN with guard rows after their end,
inputs carry NaN guard rows, and the padding slots of the last time tile of a time-tiled analysis input hold NaN and +inf.
A valid output must be finite and within the elementwise bound of `check_close`; a guard must come back bit for bit.

The analysis cases are named after the kernel they are meant to reach, and each asserts (under torch.profiler) that this
kernel is the one that ran, so that a later change of a dispatch threshold cannot move a case onto another branch
unnoticed.  `test_checker_rejects_known_defects` (no GPU) shows that the bound is tight enough to catch the defects these
kernels could plausibly have."""
import numpy as np
import pytest

from kernel_check import (GUARD, POISON, U, _note, _poisoned, _real_view, _table_K, _table_scale, _torch, _upload_rows, check_close,
                          check_guard, gamma)
from scri_b200 import _lib, _sf, plan as P
from scri_b200 import _quaternion as Q

gpu = pytest.mark.gpu


# --------------------------------------------------------------------------------------------- synthesis reference (CPU)
def _synth_reference(a, Y, off, scl, rows=None, cols=None, exact=True):
    """F = (a Y^T - c) k (per real part) and S = ((|a_r| + |a_i|)(|Y_r| + |Y_i|)^T + |c|) |k|, over the given rows and complex
    columns; in long double when `exact`, else float64 BLAS."""
    rows = slice(None) if rows is None else rows
    cols = slice(None) if cols is None else np.asarray(cols)
    ar, Yc = a[rows], Y[cols]
    if exact:
        F = ar.astype(np.clongdouble) @ Yc.astype(np.clongdouble).T
    else:
        F = ar @ Yc.T
    rc = np.arange(Y.shape[0])[cols]
    rcol = np.stack([2 * rc, 2 * rc + 1], axis=-1).ravel()
    c, k = off[rcol], scl[rcol]
    S = (np.abs(ar.real) + np.abs(ar.imag)) @ (np.abs(Yc.real) + np.abs(Yc.imag)).T
    S = (np.repeat(S, 2, axis=-1) + np.abs(c)) * np.abs(k)
    return (_real_view(F) - c) * k, S


def _synth_ref_err(K):
    return 2 * (K + 2) * U   # a float64 reference's own worst case (real GEMM of length 2K, then the epilogue)


# ---------------------------------------------------------------------------------------------- analysis reference (CPU)
def _lm_m(ell_min, ell_max):
    return np.array([m for ell in range(ell_min, ell_max + 1) for m in range(-ell, ell + 1)])


def _analysis_reference(f, E, Wt, ell_min, ell_max, exact=True):
    """a_lm = sum_j Wt[lm, j] sum_k f[j, k] E[k, m] for every row of f [N, n_theta, n_phi], and the same over absolute values."""
    N, nt, nph = f.shape
    ms = _lm_m(ell_min, ell_max)
    dt = np.clongdouble if exact else np.complex128
    Fm = (f.reshape(-1, nph).astype(dt) @ E.astype(dt)).reshape(N, nt, -1)
    SF = ((np.abs(f.real) + np.abs(f.imag)).reshape(-1, nph) @ (np.abs(E.real) + np.abs(E.imag))).reshape(N, nt, -1)
    ref = np.zeros((N, ms.size), dtype=dt)
    S = np.zeros((N, ms.size))
    Wd = Wt.astype(np.longdouble if exact else np.float64)
    for mi in range(2 * ell_max + 1):
        sel = np.nonzero(ms == mi - ell_max)[0]
        ref[:, sel] = Fm[:, :, mi] @ Wd[sel].T
        S[:, sel] = SF[:, :, mi] @ np.abs(Wt[sel]).T
    return ref, S


def _analysis_reference_at(f, E, Wt, ell_min, ell_max, t, lm):
    """Long-double a_lm at the (time, lm) pairs given."""
    ms = _lm_m(ell_min, ell_max)
    out = np.empty(t.size, dtype=np.clongdouble)
    for i in range(0, t.size, 256):
        tt, ll = t[i : i + 256], lm[i : i + 256]
        Ec = E[:, ms[ll] + ell_max].astype(np.clongdouble)                    # [k, p]
        fm = np.einsum("pjk,kp->pj", f[tt].astype(np.clongdouble), Ec)
        out[i : i + 256] = np.einsum("pj,pj->p", fm, Wt[ll].astype(np.longdouble))
    return out


# ------------------------------------------------------------------------------------------------------- CPU self-test
def test_checker_rejects_known_defects():
    """The elementwise bound accepts a correct result computed in another order and rejects a dropped k-slab of 8 modes,
    one output column shifted by one, a last partial time tile that was never written (left poisoned or zero) and one
    element off by 1e3 gamma S; a guard row that was written is caught as well."""
    rng = np.random.default_rng(5)
    N, n, G = 70, 20, 40                                   # one full 64-row tile and a partial one of 6 rows
    a = rng.normal(size=(N, n)) + 1j * rng.normal(size=(N, n))
    Y = rng.normal(size=(G, n)) + 1j * rng.normal(size=(G, n))
    off, scl = rng.normal(size=2 * G), rng.uniform(0.5, 2.0, size=2 * G) * rng.choice([-1.0, 1.0], size=2 * G)
    ref, S = _synth_reference(a, Y, off, scl)

    def synth(aa):                                         # float64, summed term by term (another order than BLAS)
        F = np.zeros((aa.shape[0], G), dtype=complex)
        for k in range(n):
            F += aa[:, k : k + 1] * Y[None, :, k]
        return (_real_view(F) - off) * scl

    good = synth(a)
    assert check_close(good, ref, S, n, "correct") < 1.0
    dropped = a.copy()
    dropped[:, 8:16] = 0.0
    with pytest.raises(AssertionError):
        check_close(synth(dropped), ref, S, n, "dropped k-slab")
    shifted = good.copy()
    shifted[:, 10:12] = good[:, 12:14]                     # complex column 5 holds column 6
    with pytest.raises(AssertionError):
        check_close(shifted, ref, S, n, "shifted column")
    for fill in (np.nan, 0.0):
        partial = good.copy()
        partial[64:] = fill
        with pytest.raises(AssertionError):
            check_close(partial, ref, S, n, "missing last tile")
    one = good.copy()
    one[37, 21] += 1e3 * gamma(n) * S[37, 21]
    with pytest.raises(AssertionError):
        check_close(one, ref, S, n, "one element")
    buf = np.zeros((N + 4, 2 * G))
    buf[N:].view(np.int64)[:] = POISON
    check_guard(buf, N, "untouched guard")
    buf[N + 3, 7] = 0.0
    with pytest.raises(AssertionError):
        check_guard(buf, N, "written guard")
    # the analysis references agree with each other (the sampled one is what the large grids are checked against)
    f = rng.normal(size=(5, 7, 9)) + 1j * rng.normal(size=(5, 7, 9))
    E, Wt = _sf.analysis_tables(-2, 1, 3, 7, 9)
    full, S = _analysis_reference(f, E, Wt, 1, 3)
    f64, _ = _analysis_reference(f, E, Wt, 1, 3, exact=False)
    check_close(f64, full, S, 16, "float64 analysis reference")
    t, lm = np.meshgrid(np.arange(5), np.arange(full.shape[1]), indexing="ij")
    assert np.array_equal(_analysis_reference_at(f, E, Wt, 1, 3, t.ravel(), lm.ravel()), full.ravel())


# ------------------------------------------------------------------------------------------------------- GPU helpers
def _kernel_names(fn):
    """Names of the CUDA kernels `fn` runs (torch.profiler, CUDA activities only), spaces removed."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name.replace(" ", "") for e in prof.events()]


def _ran(names, kernel):
    return sum(kernel.replace(" ", "") in n for n in names)


# -------------------------------------------------------------------------------------------------------------- analysis
TILED_NP = 9   # analysis.cu: the tiled kernel aliases its f_m buffer onto the tile when ell_max + 1 <= TILED_NP


def _fused_time_tile(n_theta, n_phi, ell_min, ell_max):
    """The time tile scrib200_map2salm gives its fused kernel (analysis.cu: fused_smem and the loop in scrib200_map2salm);
    0 = the DFT + quadrature fallback."""
    nm, n_modes = 2 * ell_max + 1, ell_max * (ell_max + 2) - ell_min * ell_min + 1

    def smem(T):
        return (n_phi * nm + T * n_theta * n_phi + T * n_theta * nm) * 16 + n_modes * n_theta * 8

    if smem(1) > 200 * 1024:
        return 0
    T = 1
    while T < 8 and smem(T + 1) <= 100 * 1024:
        T += 1
    return T


# id, kernels that must run, n_theta, n_phi, spin, ell_min, ell_max, environment, expectation:
#   tile = what scrib200_map2salm_tile_size returns (the case then calls scrib200_map2salm_tiled with it), alias = the tiled
#   kernel's aliasing, fused = the time tile of the time-major kernel (the case calls scrib200_map2salm), oracle = also
#   compared with oracle.spinsfast.map2salm
ANALYSIS_CASES = [
    ("persist1-ellmin0", ["map2salm_persist_kernel<1>"], 17, 17, -2, 0, 8, {}, dict(tile=8, oracle=True)),
    ("persist1-ellmin1", ["map2salm_persist_kernel<1>"], 17, 17, -1, 1, 8, {}, dict(tile=8)),
    ("persist1-ellmin2", ["map2salm_persist_kernel<1>"], 17, 17, 2, 2, 8, {}, dict(tile=8)),
    ("persist1-warps7-min", ["map2salm_persist_kernel<1>"], 13, 13, 1, 0, 6, {"SCRIB200_ANALYSIS_WARPS": "7"}, dict(tile=8)),
    ("persist1-warps17", ["map2salm_persist_kernel<1>"], 13, 13, -2, 2, 6, {"SCRIB200_ANALYSIS_WARPS": "17"}, dict(tile=8)),
    ("persist2-ellmin0", ["map2salm_persist_kernel<2>"], 19, 19, 0, 0, 9, {}, dict(tile=8)),
    ("persist2-ellmin2", ["map2salm_persist_kernel<2>"], 19, 19, -2, 2, 9, {}, dict(tile=8)),
    ("dmma1", ["map2salm_dmma_kernel<1>"], 19, 33, 1, 2, 8, {}, dict(tile=8)),
    ("dmma2-nonpersistent", ["map2salm_dmma_kernel<2>"], 19, 19, 2, 0, 9, {"SCRIB200_ANALYSIS_NONPERSISTENT": "1"}, dict(tile=8)),
    ("tiled-T8-aliased-scalar", ["map2salm_tiled_kernel<9>"], 17, 17, -1, 2, 8, {"SCRIB200_ANALYSIS_SCALAR": "1"}, dict(tile=8, alias=True)),
    ("tiled-T8-scalar", ["map2salm_tiled_kernel<9>"], 19, 19, 0, 2, 9, {"SCRIB200_ANALYSIS_SCALAR": "1"}, dict(tile=8, alias=False)),
    ("tiled-T4-aliased", ["map2salm_tiled_kernel<9>"], 33, 25, -2, 2, 8, {}, dict(tile=4, alias=True)),
    ("tiled-T4", ["map2salm_tiled_kernel<9>"], 21, 21, 1, 0, 10, {}, dict(tile=4, alias=False)),
    ("tiled-T2-aliased", ["map2salm_tiled_kernel<9>"], 67, 19, 2, 2, 8, {}, dict(tile=2, alias=True)),
    ("tiled-T2", ["map2salm_tiled_kernel<9>"], 25, 25, -1, 1, 12, {}, dict(tile=2, alias=False)),
    ("fused-T1", ["map2salm_fused_kernel"], 31, 31, -2, 2, 15, {}, dict(tile=0, fused=1)),
    ("fused-T7", ["map2salm_fused_kernel"], 19, 19, 1, 1, 9, {}, dict(fused=7)),
    ("fused-T8", ["map2salm_fused_kernel"], 9, 9, 0, 0, 4, {}, dict(fused=8, oracle=True)),
    ("dft-quad", ["map2salm_dft_kernel", "map2salm_quad_kernel"], 65, 65, 2, 2, 15, {}, dict(tile=0, fused=0)),
]
ANALYSIS_TIMES = (3001, 1, 7, 8, 9)   # 3001 > 148 SMs x 8 x 2: every persistent CTA walks several tiles through both buffers
LD_BUDGET = 1.5e8                     # multiply-adds up to which the whole reference is taken in long double


@gpu
@pytest.mark.parametrize("case", ANALYSIS_CASES, ids=[c[0] for c in ANALYSIS_CASES])
def test_map2salm_branch_vs_long_double_reference(case, monkeypatch):
    """White noise on the grid (not band limited) through the analysis branch the case names, at 1, 7, 8, 9 and 3001 time
    steps, against a_lm = sum_j Wt[lm, j] sum_k f[j, k] E[k, m] with the tables the kernel gets."""
    name, kernels, n_theta, n_phi, s, ell_min, ell_max, env, want = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    torch = _torch()
    lib = _lib.load()
    G = n_theta * n_phi
    n_modes = _sf.LM_total_size(ell_min, ell_max)
    E, Wt = _sf.analysis_tables(s, ell_min, ell_max, n_theta, n_phi)
    trig = np.ascontiguousarray(np.conj(E[:, ell_max:]))          # (cos, sin)(m phi_k) / n_phi, m = 0..ell_max
    d_E, d_Wt, d_trig = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (E, Wt, trig))
    tile = lib.scrib200_map2salm_tile_size(n_theta, n_phi, ell_min, ell_max)
    if "tile" in want:
        assert tile == want["tile"], f"{name}: scrib200_map2salm_tile_size gives {tile}"
    if "alias" in want:
        assert (ell_max + 1 <= TILED_NP) == want["alias"]
    time_major = "fused" in want
    if time_major:
        assert _fused_time_tile(n_theta, n_phi, ell_min, ell_max) == want["fused"]
    T = tile

    rng = np.random.default_rng(1000 + ANALYSIS_CASES.index(case))
    N = ANALYSIS_TIMES[0]
    f = rng.normal(size=(N, n_theta, n_phi)) + 1j * rng.normal(size=(N, n_theta, n_phi))
    K = n_theta + n_phi
    exact = N * G * (2 * ell_max + 1) + N * n_modes * n_theta <= LD_BUDGET
    ref, S = _analysis_reference(f, E, Wt, ell_min, ell_max, exact=exact)
    if not exact:   # long double at the first and last element of every 256-thread block of the quadrature kernel, and rows 0, N-1
        flat = np.unique(np.concatenate([np.arange(0, N * n_modes, 256), np.arange(255, N * n_modes, 256), [N * n_modes - 1],
                                         np.arange(n_modes), (N - 1) * n_modes + np.arange(n_modes)]))
        ref_at = _analysis_reference_at(f, E, Wt, ell_min, ell_max, flat // n_modes, flat % n_modes)

    def run(n):
        out = _poisoned((n + GUARD, 2 * n_modes))
        if time_major:
            grid = _upload_rows(f[:n].reshape(n, G), GUARD)
            ws = torch.empty(max(int(lib.scrib200_map2salm_workspace_bytes(n, n_theta, n_phi, ell_max)), 16), dtype=torch.uint8, device="cuda")
            call = lambda: _lib.check(lib.scrib200_map2salm(_lib.ptr(grid), n, n_theta, n_phi, _lib.ptr(d_E), _lib.ptr(d_Wt), ell_min, ell_max,
                                                            _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "map2salm")
        else:
            nt = -(-n // T)
            rows = np.full((nt * T, G), np.nan, dtype=complex)
            rows[:n] = f[:n].reshape(n, G)
            host = np.full((nt + 1, G, T), np.nan, dtype=complex)       # one guard tile after the input
            host[:nt] = rows.reshape(nt, T, G).transpose(0, 2, 1)       # host[b, g, tt] = f[b T + tt, g]
            pad = host[nt - 1, :, n - (nt - 1) * T :]                  # the slots of the last tile past n: NaN / +inf
            pad.real[0::2], pad.imag[1::2] = np.inf, np.inf
            grid = torch.from_numpy(_real_view(host.reshape(-1, G * T)).copy()).cuda()
            call = lambda: _lib.check(lib.scrib200_map2salm_tiled(_lib.ptr(grid), T, n, n_theta, n_phi, _lib.ptr(d_trig), _lib.ptr(d_Wt),
                                                                  ell_min, ell_max, _lib.ptr(out), _lib.stream_ptr()), "map2salm_tiled")
        return out, grid, call

    worst = 0.0
    for i, n in enumerate(ANALYSIS_TIMES):
        out, grid, call = run(n)
        grid_before = grid.cpu().numpy()
        if i == 0:
            names = _kernel_names(call)
            ran = [x for x in names if "map2salm" in x]
            for k in kernels:
                assert _ran(ran, k) == 1, f"{name}: expected {k}, the profiler saw {ran}"
            assert len(ran) == len(kernels), f"{name}: the profiler saw {ran}"
        else:
            call()
        torch.cuda.synchronize()
        o = out.cpu().numpy()
        check_guard(o, n, f"{name} n={n} output")
        assert np.array_equal(grid.cpu().numpy().view(np.int64), grid_before.view(np.int64)), f"{name}: input modified"
        got = o[:n].view(complex)
        worst = max(worst, check_close(got, ref[:n], S[:n], K, f"{name} n={n}", ref_err=0.0 if exact else 3 * (K + 4) * U))
        if not exact:
            sel = flat < n * n_modes
            fl = flat[sel]
            worst = max(worst, check_close(got.ravel()[fl][:, None], ref_at[sel][:, None], S.ravel()[fl][:, None], K, f"{name} n={n} sampled"))
    _note(f"{kernels[0]} ({name})", worst)
    if want.get("oracle"):
        from oracle import spinsfast as ospf

        assert got.shape[0] == 9 and _rel(got, ospf.map2salm(f[:9], s, ell_max)[:, ell_min**2 :]) < 1e-13


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


# ------------------------------------------------------------------------------------------------------------- synthesis
# id, entry point, selecting variable and value, kernel instantiation
SYNTH_KERNELS = [
    ("folded-v0", "folded", "SCRIB200_SYNTH_VARIANT", "0", "swsh_synth_dmma_kernel<8, 4, 64>"),
    ("folded-v1", "folded", "SCRIB200_SYNTH_VARIANT", "1", "swsh_synth_dmma_kernel<16, 3, 128>"),
    ("folded-v2", "folded", "SCRIB200_SYNTH_VARIANT", "2", "swsh_synth_dmma_kernel<16, 3, 64>"),
    ("3m-stages2", "3m", "SCRIB200_SYNTH3M_STAGES", "2", "swsh_synth3m_kernel<2>"),
    ("3m-stages3", "3m", "SCRIB200_SYNTH3M_STAGES", "3", "swsh_synth3m_kernel<3>"),
    ("3m-stages4", "3m", "SCRIB200_SYNTH3M_STAGES", "4", "swsh_synth3m_kernel<4>"),
]
# n_modes -> (spin, ell_min, ell_max) of the table
SYNTH_BANDS = {1: (0, 0, 0), 3: (0, 1, 1), 5: (1, 2, 2), 77: (-2, 2, 8), 1089: (0, 0, 32)}
SYNTH_SHAPES = [(1, 1), (5, 361), (77, 625), (1089, 361), (1089, 1), (1, 625)]
SYNTH_TIMES = (1000, 1, 63, 65, 129)
_synth_cache = {}


def _synth_problem(n_modes, G, N, seed):
    """Modes, rotor-grid table (packed as the folded kernel takes it), offset and scale, and the reference."""
    key = (n_modes, G, N, seed)
    if key not in _synth_cache:
        rng = np.random.default_rng(seed)
        s, ell_min, ell_max = SYNTH_BANDS[n_modes]
        R = Q.qnormalized(rng.normal(size=(G, 4)))
        B, Kpad, Ncpad = P.pack_synthesis_matrix(_sf.SWSH_grid(R, s, ell_max), ell_min, ell_max)
        Y = B[0 : 2 * n_modes : 2, 0 : 2 * G : 2].T + 1j * B[0 : 2 * n_modes : 2, 1 : 2 * G : 2].T   # exactly what the kernel reads
        a = rng.normal(size=(N, n_modes)) + 1j * rng.normal(size=(N, n_modes))
        off = rng.normal(size=2 * G)
        scl = rng.uniform(0.25, 4.0, size=2 * G) * rng.choice([-1.0, 1.0], size=2 * G)
        exact = N * n_modes * G <= 5e7
        ref, S = _synth_reference(a, Y, off, scl, exact=exact)
        samples = None
        if not exact:   # long double on the first and last row of every 64- and 128-row tile and column of every 32-column tile
            rows = np.unique(np.concatenate([np.arange(0, N, 64), np.arange(63, N, 64), [N - 1]]))
            cols = np.unique(np.concatenate([np.arange(0, G, 32), np.arange(31, G, 32), [G - 1]]))
            samples = (rows, _synth_reference(a, Y, off, scl, rows=rows), cols, _synth_reference(a, Y, off, scl, cols=cols))
        _synth_cache[key] = (a, B, Kpad, Ncpad, Y, off, scl, ref, S, exact, samples)
    return _synth_cache[key]


def _synth_launcher(kind, a_dev, n, n_modes, G, B, Kpad, Ncpad, d_off, d_scl, out):
    """The scrib200_swsh_synthesize(_3m) call on n rows; for the 3M kernel the table is re-laid out by
    scrib200_swsh_pack3m into a poisoned buffer first, and that layout is checked exactly."""
    torch = _torch()
    lib = _lib.load()
    d_B = torch.from_numpy(B).cuda()
    if kind == "folded":
        return lambda: _lib.check(lib.scrib200_swsh_synthesize(_lib.ptr(a_dev), n, n_modes, _lib.ptr(d_B), Kpad, Ncpad, _lib.ptr(d_off),
                                                               _lib.ptr(d_scl), G, _lib.ptr(out), _lib.stream_ptr()), "swsh_synthesize")
    npad, Gpad = -(-n_modes // 8) * 8, -(-G // 32) * 32
    d_B3 = _poisoned((3, npad, Gpad))
    _lib.check(lib.scrib200_swsh_pack3m(_lib.ptr(d_B), Kpad, Ncpad, n_modes, G, _lib.ptr(d_B3), npad, Gpad, _lib.stream_ptr()), "swsh_pack3m")
    want = np.zeros((3, npad, Gpad))
    want[0, :n_modes, :G] = B[0 : 2 * n_modes : 2, 0 : 2 * G : 2]
    want[1, :n_modes, :G] = B[0 : 2 * n_modes : 2, 1 : 2 * G : 2]
    want[2] = want[0] + want[1]
    assert np.array_equal(d_B3.cpu().numpy().view(np.int64), want.view(np.int64)), "swsh_pack3m: planes differ"
    return lambda: _lib.check(lib.scrib200_swsh_synthesize_3m(_lib.ptr(a_dev), n, n_modes, _lib.ptr(d_B3), npad, Gpad, _lib.ptr(d_off),
                                                              _lib.ptr(d_scl), G, _lib.ptr(out), _lib.stream_ptr()), "swsh_synthesize_3m")


def _synth_case(kernel, n_modes, G, times, seed, monkeypatch, expect_launches=1):
    cid, kind, var, val, kname = kernel
    monkeypatch.setenv(var, val)
    torch = _torch()
    a, B, Kpad, Ncpad, Y, off, scl, ref, S, exact, samples = _synth_problem(n_modes, G, times[0], seed)
    d_off, d_scl = _poisoned(2 * G + 64), _poisoned(2 * G + 64)   # NaN guard after the 2 G values each kernel may read
    d_off[: 2 * G] = torch.from_numpy(off).cuda()
    d_scl[: 2 * G] = torch.from_numpy(scl).cuda()
    worst = 0.0
    for i, n in enumerate(times):
        a_dev = _upload_rows(a[:n], GUARD)
        out = _poisoned((n + GUARD, 2 * G))
        call = _synth_launcher(kind, a_dev, n, n_modes, G, B, Kpad, Ncpad, d_off, d_scl, out)
        if i == 0:
            names = _kernel_names(call)
            assert _ran(names, kname) == expect_launches and len([x for x in names if "swsh_synth" in x]) == expect_launches, (cid, names)
        else:
            call()
        o = out.cpu().numpy()
        check_guard(o, n, f"{cid} n={n} output")
        got = o[:n]
        what = f"{cid} {n}x{n_modes}x{G}"
        worst = max(worst, check_close(got, ref[:n], S[:n], n_modes, what, ref_err=0.0 if exact else _synth_ref_err(n_modes)))
        if samples is not None:
            rows, (rr, rS), cols, (cr, cS) = samples
            sel = rows < n
            worst = max(worst, check_close(got[rows[sel]], rr[sel], rS[sel], n_modes, what + " sampled rows"))
            rc = np.stack([2 * cols, 2 * cols + 1], axis=-1).ravel()
            worst = max(worst, check_close(got[:, rc], cr[:n], cS[:n], n_modes, what + " sampled columns"))
    _note(kname, worst)


@gpu
@pytest.mark.parametrize("kernel", SYNTH_KERNELS, ids=[k[0] for k in SYNTH_KERNELS])
@pytest.mark.parametrize("shape", SYNTH_SHAPES, ids=[f"modes{m}-G{g}" for m, g in SYNTH_SHAPES])
def test_swsh_synthesis_kernels_vs_long_double_reference(kernel, shape, monkeypatch):
    """F = (a Y^T - c) k^w through every synthesis kernel at 1, 63, 65, 129 and 1000 time steps (partial row tiles of 64 and
    128), n_modes 1..1089 (partial k-slabs), G not a multiple of 32 or 64 (partial column tiles), per-part offset and scale."""
    n_modes, G = shape
    _synth_case(kernel, n_modes, G, SYNTH_TIMES, 7 + n_modes + G, monkeypatch)


@gpu
@pytest.mark.parametrize("kernel", SYNTH_KERNELS, ids=[k[0] for k in SYNTH_KERNELS])
def test_swsh_synthesis_band_walk(kernel, monkeypatch):
    """A table over 48 MB per band of column tiles: the CTAs walk bands (synth.cu), here with several row tiles and a last
    band narrower than the others."""
    n_modes, G, N = 1089, 2000, 300
    Kpad, npad = -(-2 * n_modes // 16) * 16, -(-n_modes // 8) * 8
    if kernel[1] == "folded":
        band, tiles, rows = (48 << 20) // (Kpad * 64 * 8), -(-2 * G // 64), -(-N // (128 if kernel[3] == "1" else 64))
    else:
        band, tiles, rows = (48 << 20) // (3 * npad * 32 * 8), -(-G // 32), -(-N // 64)
    assert band < tiles and tiles % band != 0 and rows > 1, (band, tiles, rows)
    _synth_case(kernel, n_modes, G, (N,), 17, monkeypatch)


@gpu
@pytest.mark.parametrize("kernel", [SYNTH_KERNELS[0], SYNTH_KERNELS[1], SYNTH_KERNELS[4]], ids=["folded-v0", "folded-v1", "3m-stages3"])
def test_swsh_synthesis_row_slabs(kernel, monkeypatch):
    """Past 65535 x 64 rows the synthesis goes in two launches (gridDim.y <= 65535): the rows on both sides of the slab
    boundary in long double, the whole array against a float64 reference, and exactly two kernel launches."""
    cid, kind, var, val, kname = kernel
    monkeypatch.setenv(var, val)
    torch = _torch()
    max_rows = 65535 * 64
    N, n_modes, G = max_rows + 77, 3, 8
    rng = np.random.default_rng(41)
    s, ell_min, ell_max = SYNTH_BANDS[n_modes]
    B, Kpad, Ncpad = P.pack_synthesis_matrix(_sf.SWSH_grid(Q.qnormalized(rng.normal(size=(G, 4))), s, ell_max), ell_min, ell_max)
    Y = B[0 : 2 * n_modes : 2, 0 : 2 * G : 2].T + 1j * B[0 : 2 * n_modes : 2, 1 : 2 * G : 2].T
    a = rng.normal(size=(N, n_modes)) + 1j * rng.normal(size=(N, n_modes))
    off = rng.normal(size=2 * G)
    scl = rng.uniform(0.25, 4.0, size=2 * G)
    d_off, d_scl = torch.from_numpy(off).cuda(), torch.from_numpy(scl).cuda()
    a_dev = _upload_rows(a, GUARD)
    out = _poisoned((N + GUARD, 2 * G))
    call = _synth_launcher(kind, a_dev, N, n_modes, G, B, Kpad, Ncpad, d_off, d_scl, out)
    names = _kernel_names(call)
    assert _ran(names, kname) == 2 and len([x for x in names if "swsh_synth" in x]) == 2, names
    del a_dev
    o = out.cpu().numpy()
    del out
    check_guard(o, N, f"{cid} output")
    lo = max_rows - 128
    rr, rS = _synth_reference(a, Y, off, scl, rows=np.arange(lo, N))
    worst = check_close(o[lo:N], rr, rS, n_modes, f"{cid} rows {lo}..{N} (slab boundary {max_rows})")
    for r0 in range(0, N, 1 << 20):
        r1 = min(N, r0 + (1 << 20))
        rr, rS = _synth_reference(a, Y, off, scl, rows=np.arange(r0, r1), exact=False)
        worst = max(worst, check_close(o[r0:r1], rr, rS, n_modes, f"{cid} rows {r0}..{r1}", ref_err=_synth_ref_err(n_modes)))
    _note(kname, worst)


# ------------------------------------------------------------------------------------------------------ synthesis table
def _pack_grid(kind, n_theta, n_phi):
    if kind == "regular":   # spinsfast's grid: theta inclusive (the first and last rings are the poles), phi half open
        th, ph = np.meshgrid(np.linspace(0.0, np.pi, n_theta), np.linspace(0.0, 2 * np.pi, n_phi, endpoint=False), indexing="ij")
        return Q.from_spherical_coords(th.ravel(), ph.ravel())
    R, _ = P.boosted_rotor_grid(Q.qnormalized(np.array([1.0, 2.0, 3.0, 4.0])), np.array([0.1, -0.2, 0.3]), n_theta, n_phi)
    return R.reshape(-1, 4)


# spin, ell_min, ell_max, table_ell_max, grid, n_theta, n_phi
PACK_CASES = [
    (-2, 0, 8, 8, "regular", 17, 17),
    (-2, 3, 12, 15, "boosted", 13, 11),
    (-1, 1, 32, 32, "regular", 9, 8),
    (-1, 2, 20, 24, "boosted", 11, 9),
    (0, 0, 32, 34, "boosted", 7, 9),
    (0, 1, 16, 16, "regular", 33, 33),
    (1, 1, 9, 12, "regular", 19, 19),
    (1, 0, 5, 5, "boosted", 11, 11),
    (2, 2, 32, 33, "regular", 13, 7),
    (2, 3, 16, 20, "boosted", 17, 17),
]


def _pack_reference(s, ell_min, ell_max, Lt, R):
    from oracle import sf as osf

    B, Kpad, Ncpad = P.pack_synthesis_matrix(osf.SWSH_grid(R, s, ell_max), ell_min, ell_max)
    sc = np.zeros((R.shape[0], (ell_max + 1) ** 2))
    sc[:, ell_min**2 :] = _table_scale(R, s, ell_min, ell_max, Lt)
    SB, _, _ = P.pack_synthesis_matrix(sc * (1 + 1j), ell_min, ell_max)
    return B, np.abs(SB), Kpad, Ncpad


def test_table_scale_bounds_the_host_recurrence():
    """The table bound holds for the host's own float64 recurrence (_sf.SWSH_grid, the algorithm the device kernel runs)
    against the oracle's long-double Wigner sums, and rejects a 1e-6 relative change in one small element near a pole."""
    s, ell_min, ell_max = 2, 2, 20
    R = _pack_grid("regular", 11, 9)
    B, SB, Kpad, Ncpad = _pack_reference(s, ell_min, ell_max, ell_max, R)
    host, _, _ = P.pack_synthesis_matrix(_sf.SWSH_grid(R, s, ell_max), ell_min, ell_max)
    K = _table_K(ell_max)
    assert check_close(host, B, SB, K, "host table") < 0.5
    i = _sf.LM_index(ell_max, -ell_max + 1, ell_min)
    g = 9 + 3                                            # second ring, next to the north pole: a tiny, high-l element
    assert 0.0 < abs(B[2 * i, 2 * g]) < 1e-6
    bad = host.copy()
    bad[2 * i, 2 * g] *= 1 + 1e-6
    with pytest.raises(AssertionError):
        check_close(bad, B, SB, K, "one small element")


@gpu
@pytest.mark.parametrize("case", PACK_CASES, ids=[f"s{c[0]}-lmin{c[1]}-L{c[2]}-Lt{c[3]}-{c[4]}{c[5]}x{c[6]}" for c in PACK_CASES])
def test_swsh_pack_vs_oracle_wigner(case):
    """The device-built synthesis table (scrib200_swsh_pack, into a NaN-poisoned buffer) against the packed oracle SWSH_grid,
    element by element, and its Kpad / Ncpad padding exactly zero."""
    from scri_b200 import ops

    s, ell_min, ell_max, Lt, kind, n_theta, n_phi = case
    torch = _torch()
    lib = _lib.load()
    R = _pack_grid(kind, n_theta, n_phi)
    G = R.shape[0]
    B, SB, Kpad, Ncpad = _pack_reference(s, ell_min, ell_max, Lt, R)
    seed_d, _, uv_d = ops.wigner_tables_device(Lt)
    d_R = torch.from_numpy(np.ascontiguousarray(R)).cuda()
    d_B = _poisoned((Kpad, Ncpad))
    _lib.check(lib.scrib200_swsh_pack(_lib.ptr(d_R), G, s, ell_min, ell_max, _lib.ptr(seed_d), _lib.ptr(uv_d), Lt, _lib.ptr(d_B), Kpad, Ncpad,
                                      _lib.stream_ptr()), "swsh_pack")
    got = d_B.cpu().numpy()
    n = _sf.LM_total_size(ell_min, ell_max)
    assert np.array_equal(got[2 * n :], np.zeros_like(got[2 * n :])) and np.array_equal(got[:, 2 * G :], np.zeros_like(got[:, 2 * G :]))
    assert not np.signbit(got[2 * n :]).any() and not np.signbit(got[:, 2 * G :]).any()
    _note("swsh_pack_kernel", check_close(got, B, SB, _table_K(ell_max), f"swsh_pack s={s} ell=[{ell_min}, {ell_max}] Lt={Lt} {kind}"))
