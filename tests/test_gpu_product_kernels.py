"""Every launch branch of the fused mode product (product.cu: scrib200_modes_product, K9), the separable theta stages
(scrib200_theta_synth / scrib200_theta_quad, K11) and the pointwise grid product (mix.cu: scrib200_grid_product) against a
plain long-double reference of the same operation, through the C ABI.

The references take the float64 tables the kernels receive (`_product._lambda`, `_sf.analysis_tables`) and write each
operation out literally:
  K9             F^i_m(j) = sum_l lambda^i_lm(j) a^i_lm,   P_M(j) = sum_{m1 + m2 = M (mod n_phi)} F^1_m1(j) F^2_m2(j),
                 out_lM = sum_j W_lM(j) P_M(j)  (the alias condition as a true modulo condition, not the kernel's qmax);
  theta_synth    out[t, j, m] = sum_l lambda_lm(theta_j) a_lm;
  theta_quad     out[t, lm] = sum_j W_lM(theta_j) P[t, j, M];
  grid_product   out = a b.
Each valid output must be finite and within |out - ref| <= gamma(K) S (kernel_check.py), S the same chain over absolute
values.  Outputs start poisoned with guard rows after them, which must come back bit for bit; inputs carry NaN guard rows.

The persistent kernels stride over groups of 4 time steps; the long runs (K9: 1187 steps, K11: 2371) give every CTA at least
two turns and end on a partial group, and K9 also runs with 1, 3 and 4 CTAs (pairs for the cluster kernel).  Each case
asserts from the host tables the branch it is meant to reach (alias terms qmax, ring chunks, staged or direct output
store), so that a later table change cannot move it off its branch unnoticed; which kernel instantiation runs is checked
under torch.profiler in a child process."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest

from kernel_check import (GUARD, POISON, U, _note, _poisoned, _table_K, _table_scale, _torch, _upload_rows, check_close, check_guard,
                          gamma)
from scri_b200 import _lib, _product, _sf

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LD_BUDGET = 1.5e8   # multiply-adds up to which the whole reference is taken in long double
PRODUCT_T = 4       # product.cu: time steps per CTA pass
K9_CTAS, K11_CTAS = 148, 296   # the default grid of modes_product (pairs: half of it) and the grid cap of the theta kernels


# ------------------------------------------------------------------------------------------------------ references (CPU)
def _lm_m(ell_min, ell_max):
    return np.array([m for ell in range(ell_min, ell_max + 1) for m in range(-ell, ell + 1)], dtype=int)


def _theta_contract(a, lam, ms, ell, exact):
    """F[t, j, m + ell] = sum over the stored l of lam[j, lm] a[t, lm] (a [N, n], lam [n_theta, n], ms [n] the m of every
    stored mode), and the same over absolute values, |a| = |Re| + |Im|."""
    N, nth = a.shape[0], lam.shape[0]
    F = np.zeros((N, nth, 2 * ell + 1), dtype=np.clongdouble if exact else complex)
    SF = np.zeros((N, nth, 2 * ell + 1))
    absa = np.abs(a.real) + np.abs(a.imag)
    for m in range(-ell, ell + 1):
        sel = np.nonzero(ms == m)[0]
        if sel.size == 0:
            continue
        L = lam[:, sel].T
        F[:, :, m + ell] = a[:, sel].astype(np.clongdouble) @ L.astype(np.longdouble) if exact else a[:, sel] @ L
        SF[:, :, m + ell] = absa[:, sel] @ np.abs(L)
    return F, SF


def _m_convolve(F1, F2):
    """Linear convolution over m: Pext[..., m1 + m2 + ell1 + ell2] = sum F1[..., m1 + ell1] F2[..., m2 + ell2]."""
    n1, n2 = F1.shape[-1], F2.shape[-1]
    out = np.zeros(F1.shape[:-1] + (n1 + n2 - 1,), dtype=np.result_type(F1, F2))
    for i in range(n1):
        out[..., i : i + n2] += F1[..., i : i + 1] * F2
    return out


def _fold_sets(ell1, ell2, L_out, n_phi):
    """For every output M, the indices Mp + ell1 + ell2 of the linear convolution with Mp = M (mod n_phi)."""
    Mp = np.arange(-(ell1 + ell2), ell1 + ell2 + 1)
    return [np.nonzero((Mp - M) % n_phi == 0)[0] for M in range(-L_out, L_out + 1)]


def _pairs_per_output(ell1, ell2, L_out, n_phi):
    """The number of (m1, m2) pairs each output M receives."""
    m1 = np.arange(-ell1, ell1 + 1)
    per_Mp = np.array([np.count_nonzero(np.abs(Mp - m1) <= ell2) for Mp in range(-(ell1 + ell2), ell1 + ell2 + 1)])
    return np.array([per_Mp[s].sum() for s in _fold_sets(ell1, ell2, L_out, n_phi)])


def _quadrature(P, SP, W, ms, L, exact):
    """out[t, lm] = sum_j W[lm, j] P[t, j, m + L] (rows of W in the output's order, ms their m), and over absolute values."""
    N = P.shape[0]
    out = np.zeros((N, W.shape[0]), dtype=np.clongdouble if exact else complex)
    S = np.zeros((N, W.shape[0]))
    for M in range(-L, L + 1):
        sel = np.nonzero(ms == M)[0]
        if sel.size == 0:
            continue
        Wm = W[sel].T
        out[:, sel] = P[:, :, M + L].astype(np.clongdouble) @ Wm.astype(np.longdouble) if exact else P[:, :, M + L] @ Wm
        S[:, sel] = SP[:, :, M + L] @ np.abs(Wm)
    return out, S


def _k9_tables(case):
    """The float64 tables of a K9 case, exactly as the kernel's fragments are built from them."""
    s1, l1min, l1, s2, l2min, l2, n_theta, n_phi, L_out = case
    _, Wt = _sf.analysis_tables(s1 + s2, 0, L_out, n_theta, n_phi)
    return dict(lam1=_product._lambda(s1, l1, n_theta)[:, l1min**2 :], ms1=_lm_m(l1min, l1),
                lam2=_product._lambda(s2, l2, n_theta)[:, l2min**2 :], ms2=_lm_m(l2min, l2), W=Wt, msW=_lm_m(0, L_out),
                fold=_fold_sets(l1, l2, L_out, n_phi), ell1=l1, ell2=l2, L_out=L_out,
                K=(l1 + 1) + (l2 + 1) + int(_pairs_per_output(l1, l2, L_out, n_phi).max()) + n_theta)


def _k9_reference(tab, a1, a2, exact=True):
    """Modes of the product, [N, (L_out + 1)^2], and S."""
    F1, S1 = _theta_contract(a1, tab["lam1"], tab["ms1"], tab["ell1"], exact)
    F2, S2 = _theta_contract(a2, tab["lam2"], tab["ms2"], tab["ell2"], exact)
    Pe, SPe = _m_convolve(F1, F2), _m_convolve(S1, S2)
    P = np.stack([Pe[..., idx].sum(axis=-1) for idx in tab["fold"]], axis=-1)
    SP = np.stack([SPe[..., idx].sum(axis=-1) for idx in tab["fold"]], axis=-1)
    return _quadrature(P, SP, tab["W"], tab["msW"], tab["L_out"], exact)


def _k9_cost(tab, N):
    n_theta = tab["W"].shape[1]
    return N * n_theta * (tab["ms1"].size + tab["ms2"].size + (2 * tab["ell1"] + 1) * (2 * tab["ell2"] + 1) + tab["msW"].size)


def _ref_err(K):
    return 3 * (K + 4) * U   # a float64 reference's own worst case (three stages with complex rounding)


def _sample_rows(N, grids, always=()):
    """Rows for the long-double checks of a float64-referenced run: every row of the first group and of the last (partial)
    group, and for every CTA of each grid one row of the group of its last turn (the slot in the group rotates with the CTA,
    so all four slots are covered)."""
    n_tg = -(-N // PRODUCT_T)
    rows = set(range(min(N, PRODUCT_T))) | set(range((n_tg - 1) * PRODUCT_T, N)) | {r for r in always if r < N}
    for grid in grids:
        grid = min(grid, n_tg)
        for b in range(grid):
            g = b + grid * ((n_tg - 1 - b) // grid)
            r = g * PRODUCT_T + b % PRODUCT_T
            rows.add(r if r < N else g * PRODUCT_T)
    return np.array(sorted(rows))


def _check_rows(got, ref, S, K, what, ref_err=0.0, block=256):
    """check_close over blocks of rows (bounded memory on the large outputs)."""
    worst = 0.0
    for r0 in range(0, got.shape[0], block):
        r1 = min(got.shape[0], r0 + block)
        worst = max(worst, check_close(got[r0:r1], ref[r0:r1], S[r0:r1], K, f"{what} rows {r0}..{r1}", ref_err=ref_err))
    return worst


# ---------------------------------------------------------------------------------------------------------------- cases
# id: (s1, ell1_min, ell1, s2, ell2_min, ell2, n_theta, n_phi, L_out), expected alias terms qmax, expected staged output store
K9_CASES = {
    "default": ((2, 2, 4, -1, 0, 3, 15, 15, 4), 0, True),
    "direct-store": ((0, 0, 12, 2, 2, 8, 41, 41, 20), 0, False),
    "alias-q2": ((2, 0, 10, -2, 0, 10, 11, 11, 4), 2, True),
    "alias-rect-q2": ((2, 0, 8, -2, 0, 8, 17, 9, 8), 2, True),
    "few-rings-q1": ((0, 0, 2, 0, 0, 2, 5, 5, 2), 1, True),
    "rings-mult8-Lout0": ((1, 0, 6, 1, 0, 6, 24, 29, 0), 0, True),   # l = 0 < |s1 + s2|: S = 0, the output must be exactly 0
    "rings-mult8-Lout0-s0": ((1, 0, 6, -1, 0, 6, 24, 29, 0), 0, True),   # the same with a nonzero l = 0 mode
    "Lout-above-sum": ((0, 0, 3, 0, 0, 3, 7, 15, 8), 0, False),
    "config4": ((2, 0, 32, -2, 0, 32, 129, 129, 32), 0, True),
    "below-spin": ((2, 0, 5, -2, 0, 4, 13, 13, 6), 1, True),       # l < |s| slots hold random values; lambda is zero there
    "same-buffer": ((1, 0, 6, 1, 0, 6, 17, 17, 6), 1, True),        # a1 and a2 are one device buffer (f x f)
}
K9_SHAPES = {0: "modes_product_kernel<5,11,9,512>", 1: "modes_product_kernel<9,21,18,256>", 2: "modes_product_cluster_kernel<5,12,9>"}
K9_SMALL = (1, 3, 4, 5)
K9_CTAS_N, K9_CTAS_VARIANTS = 38, (1, 3, 4)   # CTAs (pairs for the cluster kernel) at 38 steps: 10 groups, several turns each
K9_LONG = 4 * K9_CTAS * 2 + 3                 # 1187: every CTA takes two turns or more, the last group holds 3 steps
CONFIG4_LONG, CONFIG4_CTAS = 301, 7           # config4: a CPU reference at 1187 steps costs too much; 7 CTAs take 10-11 turns

# (s, ell_min, L, n_theta, n_phi of the analysis grid)
THETA_CASES = [(-2, 0, 8, 17, 17), (2, 2, 12, 24, 31), (1, 0, 16, 37, 37), (0, 3, 20, 41, 47), (-1, 0, 32, 65, 65), (2, 2, 32, 129, 96)]
K11_TIMES = (4 * K11_CTAS * 2 + 3, 1, 3, 4, 5)   # 2371: two turns of 296 CTAs or more, a partial last group


def _k9_rows(case_id):
    return (CONFIG4_LONG, CONFIG4_CTAS) if case_id == "config4" else (K9_LONG, 0)


def _k9_inputs(case_id, N):
    (s1, l1min, l1, s2, l2min, l2, *_), _, _ = K9_CASES[case_id]
    rng = np.random.default_rng(900 + list(K9_CASES).index(case_id))
    mk = lambda lmin, l: rng.normal(size=(N, (l + 1) ** 2 - lmin**2)) + 1j * rng.normal(size=(N, (l + 1) ** 2 - lmin**2))
    a1 = mk(l1min, l1)
    return a1, (a1 if case_id == "same-buffer" else mk(l2min, l2))


_k9_cache = {}


def _k9_problem(case_id):
    """Inputs, tables and reference of a K9 case at its longest run (the shorter runs use its first rows).  Long double
    throughout when affordable; otherwise a float64 reference plus long double on the sampled rows (every column of them,
    so the first and last tile of every M are included) and on the rows of the 38-step runs."""
    if case_id not in _k9_cache:
        case = K9_CASES[case_id][0]
        N, n_ctas = _k9_rows(case_id)
        a1, a2 = _k9_inputs(case_id, N)
        tab = _k9_tables(case)
        exact = _k9_cost(tab, N) <= LD_BUDGET
        ref, S = _k9_reference(tab, a1, a2, exact=exact)
        samples = None
        if not exact:
            rows = _sample_rows(N, (n_ctas or K9_CTAS, (n_ctas or K9_CTAS) // 2), always=range(K9_CTAS_N))
            samples = (rows,) + _k9_reference(tab, a1[rows], a2[rows])
        _k9_cache[case_id] = (a1, a2, tab, ref, S, exact, samples)
    return _k9_cache[case_id]


# ------------------------------------------------------------------------------------------------------- CPU self-tests
def _swap_M_groups(out, L_out, GM):
    """The outputs of the first two groups of GM consecutive M exchanged (a convolution warp writing another group's P)."""
    bad = out.copy()
    for k in range(GM):
        M, Mq = -L_out + k, -L_out + GM + k
        if Mq > L_out:
            break
        for l in range(max(abs(M), abs(Mq)), L_out + 1):
            i, j = l * (l + 1) + M, l * (l + 1) + Mq
            bad[:, [i, j]] = out[:, [j, i]]
    return bad


def test_checker_rejects_product_defects():
    """The numpy emulation of product.cu (tests/product_emulator.py, driven by the same host tables) passes the checker
    for every small case and every kernel shape, which also shows that the modulo-condition reference is the operation the
    tables encode.  On `alias-q2` the checker rejects an emulation without the alias terms (qmax 0), one without the last
    ring chunk, two M groups swapped, a partial last time group left at zero or poisoned, and one element off by 1e3 gamma S;
    a written guard word is caught as well.  The float64 references agree with the long-double ones within ref_err."""
    from product_emulator import emulate

    N = 5                                                   # a full group of 4 steps and a partial one
    for cid, (case, qmax, _) in K9_CASES.items():
        if cid == "config4":
            continue
        a1, a2 = _k9_inputs(cid, N)
        tab = _k9_tables(case)
        ref, S = _k9_reference(tab, a1, a2)
        for shape in (0, 1, 2):
            tb = _product.product_tables(*case, shape=shape)
            assert tb.fits and int(tb.cfg[5]) == qmax, (cid, shape)
            assert check_close(emulate(tb, a1, a2), ref, S, tab["K"], f"emulated {cid} shape {shape}") < 1.0
        f64, _ = _k9_reference(tab, a1, a2, exact=False)
        check_close(f64, ref, S, tab["K"], f"float64 reference {cid}", ref_err=_ref_err(tab["K"]))

    cid = "alias-q2"
    case = K9_CASES[cid][0]
    a1, a2 = _k9_inputs(cid, N)
    tab = _k9_tables(case)
    ref, S = _k9_reference(tab, a1, a2)
    K = tab["K"]
    tb = _product.product_tables(*case, shape=0)
    good = emulate(tb, a1, a2)
    for i, v in ((5, 0), (4, int(tb.cfg[4]) - 1)):          # no alias terms; the last ring chunk dropped
        bad_tb = copy.copy(tb)
        bad_tb.cfg = tb.cfg.copy()
        bad_tb.cfg[i] = v
        with pytest.raises(AssertionError):
            check_close(emulate(bad_tb, a1, a2), ref, S, K, f"cfg[{i}] = {v}")
    with pytest.raises(AssertionError):
        check_close(_swap_M_groups(good, case[8], int(tb.cfg[12])), ref, S, K, "swapped M groups")
    for fill in (0.0, np.nan):
        partial = good.copy()
        partial[4:] = fill
        with pytest.raises(AssertionError):
            check_close(partial, ref, S, K, "partial group not written")
    one = good.copy()
    i = (3, int(np.nonzero((S[3] > 0) & (S[3] < np.median(S[3])))[0][0]))   # a small element
    one[i] += 1e3 * gamma(K) * S[i]
    with pytest.raises(AssertionError):
        check_close(one, ref, S, K, "one element")
    buf = np.zeros((N + GUARD, 2 * ref.shape[1]))
    buf[N:].view(np.int64)[:] = POISON
    check_guard(buf, N, "untouched guard")
    buf[N + 1, 3] = 0.0
    with pytest.raises(AssertionError):
        check_guard(buf, N, "written guard")

    # theta references: float64 against long double, and a dropped ring of the quadrature is rejected
    rng = np.random.default_rng(3)
    s, lmin, L, nth, nph = THETA_CASES[2]
    a = rng.normal(size=(6, (L + 1) ** 2 - lmin**2)) + 1j * rng.normal(size=(6, (L + 1) ** 2 - lmin**2))
    lam = _product._lambda(s, L, nth)[:, lmin**2 :]
    F, SF = _theta_contract(a, lam, _lm_m(lmin, L), L, True)
    F64, _ = _theta_contract(a, lam, _lm_m(lmin, L), L, False)
    check_close(F64.reshape(6, -1), F.reshape(6, -1), SF.reshape(6, -1), L + 1 - lmin, "float64 theta_synth reference",
                ref_err=_ref_err(L + 1 - lmin))
    P = rng.normal(size=(6, nth, 2 * L + 1)) + 1j * rng.normal(size=(6, nth, 2 * L + 1))
    W = _sf.analysis_tables(s, 0, L, nth, nph)[1][lmin**2 :]
    q, Sq = _quadrature(P, np.abs(P.real) + np.abs(P.imag), W, _lm_m(lmin, L), L, True)
    q64, _ = _quadrature(P, np.abs(P.real) + np.abs(P.imag), W, _lm_m(lmin, L), L, False)
    check_close(q64, q, Sq, nth, "float64 theta_quad reference", ref_err=_ref_err(nth))
    P2 = P.copy()
    P2[:, nth // 2] = 0.0
    with pytest.raises(AssertionError):
        check_close(_quadrature(P2, np.abs(P2.real) + np.abs(P2.imag), W, _lm_m(lmin, L), L, False)[0], q, Sq, nth, "dropped ring")


def test_lambda_table_vs_long_double_wigner():
    """_product._lambda (the host's float64 recurrence, the lambda_lm(theta_j) of every K9 / theta_synth fragment) against
    the oracle's long-double Wigner path, elementwise with the table bound of test_gpu_swsh_kernels.py, for l <= 32 on
    spinsfast's rings with both poles."""
    from oracle import sf as osf

    L, n_theta = 32, 13
    theta = np.pi * np.arange(n_theta) / (n_theta - 1)
    R = np.stack([np.cos(theta / 2), np.zeros_like(theta), np.sin(theta / 2), np.zeros_like(theta)], axis=-1)
    worst = 0.0
    for s in (-2, -1, 0, 1, 2):
        lam = _product._lambda(s, L, n_theta)
        ref = osf.SWSH_grid(R, s, L)
        assert np.abs(ref.imag).max() <= 1e-15 * np.abs(ref.real).max()
        worst = max(worst, check_close(lam, ref.real, _table_scale(R, s, 0, L, L), _table_K(L), f"_lambda s={s}"))
        # at a pole only m = -s (north) or m = s (south) survives; the south ring is at cos(theta / 2) = 6e-17, not 0
        for j, m, tol in ((0, -s, 0.0), (n_theta - 1, s, 1e-13)):
            keep = np.array([mm == m for ell in range(L + 1) for mm in range(-ell, ell + 1)])
            assert np.abs(lam[j, ~keep]).max() <= tol and np.all(np.abs(lam[j, keep]) > 0.1), (s, j)
    assert worst < 1.0


# ------------------------------------------------------------------------------------------------------- GPU: K9
def _k9_device_tables(tb):
    torch = _torch()
    return {k: torch.from_numpy(np.ascontiguousarray(getattr(tb, k))).cuda() for k in ("perm1", "perm2", "ctl", "lamfrag", "tiles", "wtfrag")}


def _k9_launch(tb, dev, d1, n1, d2, n2, N, out, n_ctas=0, cfg=None):
    import ctypes

    lib = _lib.load()
    cfg = np.ascontiguousarray(tb.cfg if cfg is None else cfg, dtype=np.int32)
    _lib.check(
        lib.scrib200_modes_product(
            _lib.ptr(d1), n1, _lib.ptr(d2), n2, N, _lib.ptr(dev["perm1"]), _lib.ptr(dev["perm2"]), _lib.ptr(dev["ctl"]), tb.n_ctl,
            _lib.ptr(dev["lamfrag"]), dev["lamfrag"].shape[1], _lib.ptr(dev["tiles"]), tb.n_tiles_arg, _lib.ptr(dev["wtfrag"]),
            dev["wtfrag"].shape[1], cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(out), n_ctas, _lib.stream_ptr()),
        "modes_product")


def _k9_run(tb, dev, a1, a2, same, n_ctas=0, cfg=None):
    """One launch on fresh buffers: NaN guard rows after the inputs, a poisoned output with guard rows; returns the valid
    complex rows after checking the guards and that the inputs are unchanged."""
    torch = _torch()
    N = a1.shape[0]
    d1 = _upload_rows(a1, GUARD)
    d2 = d1 if same else _upload_rows(a2, GUARD)
    before = [d.cpu().numpy() for d in (d1, d2)]
    out = _poisoned((N + GUARD, 2 * tb.n_out))
    _k9_launch(tb, dev, d1, a1.shape[1], d2, a2.shape[1], N, out, n_ctas, cfg)
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    check_guard(o, N, f"modes_product N={N} output")
    for d, b in zip((d1, d2), before):
        assert np.array_equal(d.cpu().numpy().view(np.int64), b.view(np.int64)), "modes_product: input modified"
    return o[:N].view(complex)


@gpu
@pytest.mark.parametrize("shape", list(K9_SHAPES), ids=[f"shape{s}" for s in K9_SHAPES])
@pytest.mark.parametrize("case_id", list(K9_CASES))
def test_modes_product_branch_vs_long_double_reference(case_id, shape):
    """K9 through one kernel shape on white-noise factors at 1, 3, 4 and 5 steps, at 38 steps with the default grid and
    with 1, 3 and 4 CTAs (pairs), and at 1187 steps (config4: 301 steps on 7 CTAs).  The output is the same bit for bit
    for every grid, and a row is the same whether computed inside a long launch or alone."""
    case, qmax, stage_out = K9_CASES[case_id]
    tb = _product.product_tables(*case, shape=shape)
    assert tb.fits, (case_id, shape, tb.smem_bytes)
    cfg = [int(x) for x in tb.cfg]
    n_theta, L_out = case[6], case[8]
    assert cfg[5] == qmax, f"{case_id}: qmax {cfg[5]}"
    assert cfg[4] == -(-n_theta // 8)
    assert (cfg[15] == 1) == (shape == 2)
    if shape != 2:
        assert (8 * tb.n_out <= cfg[6]) == stage_out, f"{case_id}: staged output store {8 * tb.n_out} <= {cfg[6]}"
    if case_id == "config4":
        assert tb.smem_bytes == {0: 231768, 1: 231884, 2: 222144}[shape]
    same = case_id == "same-buffer"
    kname = K9_SHAPES[shape]
    dev = _k9_device_tables(tb)
    a1, a2, tab, ref, S, exact, samples = _k9_problem(case_id)
    K = tab["K"]
    ref_err = 0.0 if exact else _ref_err(K)
    N_long, n_ctas_long = _k9_rows(case_id)
    if shape == 2 and n_ctas_long:
        n_ctas_long *= 2                                    # 7 pairs: n_ctas / 2 pairs for the cluster kernel
    scale = 2 if shape == 2 else 1
    worst = 0.0

    def check(got, n, what):
        w = check_close(got, ref[:n], S[:n], K, f"{case_id} {kname} {what}", ref_err=ref_err)
        if samples is not None:
            rows, rr, rS = samples
            sel = rows < n
            w = max(w, check_close(got[rows[sel]], rr[sel], rS[sel], K, f"{case_id} {kname} {what} sampled rows"))
        return w

    single = {}
    for n in K9_SMALL:
        got = _k9_run(tb, dev, a1[:n], a2[:n], same)
        worst = max(worst, check(got, n, f"N={n}"))
        if n == 1:
            single[0] = got[0]
    runs = {}
    for c in (0,) + K9_CTAS_VARIANTS:
        runs[c] = _k9_run(tb, dev, a1[:K9_CTAS_N], a2[:K9_CTAS_N], same, n_ctas=scale * c)
        worst = max(worst, check(runs[c], K9_CTAS_N, f"N={K9_CTAS_N} n_ctas={scale * c}"))
        assert np.array_equal(runs[c].view(np.int64), runs[0].view(np.int64)), f"{case_id}: n_ctas={scale * c} differs from the default grid"
    long = _k9_run(tb, dev, a1, a2, same, n_ctas=n_ctas_long)
    worst = max(worst, check(long, N_long, f"N={N_long} n_ctas={n_ctas_long}"))
    assert np.array_equal(long[:K9_CTAS_N].view(np.int64), runs[0].view(np.int64)), f"{case_id}: rows differ between launches"
    for r in (1, 2, 3, N_long - 1):                         # every slot of a group, and the partial last group
        single[r] = _k9_run(tb, dev, a1[r : r + 1], a2[r : r + 1], same)[0]
    for r, row in single.items():
        assert np.array_equal(long[r].view(np.int64), row.view(np.int64)), f"{case_id}: row {r} differs when computed alone"
    if case_id == "below-spin":                             # the l < |s| slots of both factors must not matter
        z1, z2 = a1[:9].copy(), a2[:9].copy()
        z1[:, : case[0] ** 2], z2[:, : case[3] ** 2] = 0.0, 0.0
        assert np.array_equal(_k9_run(tb, dev, z1, z2, same), long[:9])
    _note(f"{kname}", worst)


@gpu
def test_modes_product_negative_controls():
    """alias-q2 launched without its alias terms (cfg[5] = 0) and without its last ring chunk (cfg[4] - 1): the kernel reads
    and writes less, and the checker rejects both results."""
    case_id = "alias-q2"
    case = K9_CASES[case_id][0]
    tb = _product.product_tables(*case, shape=0)
    dev = _k9_device_tables(tb)
    a1, a2, tab, ref, S, exact, _ = _k9_problem(case_id)
    n = 5
    assert exact and check_close(_k9_run(tb, dev, a1[:n], a2[:n], False), ref[:n], S[:n], tab["K"], "unmodified") < 1.0
    for i, v in ((5, 0), (4, int(tb.cfg[4]) - 1)):
        cfg = tb.cfg.copy()
        cfg[i] = v
        got = _k9_run(tb, dev, a1[:n], a2[:n], False, cfg=cfg)
        with pytest.raises(AssertionError):
            check_close(got, ref[:n], S[:n], tab["K"], f"cfg[{i}] = {v}")


# ------------------------------------------------------------------------------------------------------- GPU: K11
def _theta_synth_run(tb, dev, a):
    import ctypes

    torch = _torch()
    lib = _lib.load()
    N, n = a.shape
    d = _upload_rows(a, GUARD)
    before = d.cpu().numpy()
    out = _poisoned((N + GUARD, 2 * tb.cfg[0] * tb.nm))
    _lib.check(lib.scrib200_theta_synth(_lib.ptr(d), n, N, _lib.ptr(dev["perm"]), _lib.ptr(dev["ctl"]), tb.n_ctl, _lib.ptr(dev["lamfrag"]),
                                        dev["lamfrag"].shape[1], tb.cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(out), _lib.stream_ptr()),
               "theta_synth")
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    check_guard(o, N, f"theta_synth N={N} output")
    assert np.array_equal(d.cpu().numpy().view(np.int64), before.view(np.int64)), "theta_synth: input modified"
    return o[:N].view(complex)


@gpu
@pytest.mark.parametrize("case", THETA_CASES, ids=[f"s{c[0]}-lmin{c[1]}-L{c[2]}-{c[3]}rings" for c in THETA_CASES])
def test_theta_synth_vs_long_double_reference(case):
    """theta_synth at 2371, 1, 3, 4 and 5 steps: ring counts that are and are not multiples of 8, nm = 33 (the lane loop
    over m runs twice) and 65, and L = 32, the largest band limit whose tables fit the 113 KB of two CTAs per SM."""
    torch = _torch()
    s, lmin, L, n_theta, _ = case
    tb = _product.theta_tables(s, lmin, L, n_theta)
    assert tb.fits and tb.nm == 2 * L + 1 and int(tb.cfg[2]) == -(-n_theta // 8)
    if L == 32:
        assert tb.smem_bytes == {0: 112048, 2: 111828}[lmin], tb.smem_bytes
        assert not _product.theta_tables(s, lmin, 33, n_theta).fits
    dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(tb, k))).cuda() for k in ("perm", "ctl", "lamfrag")}
    rng = np.random.default_rng(70 + THETA_CASES.index(case))
    N = K11_TIMES[0]
    n = (L + 1) ** 2 - lmin**2
    a = rng.normal(size=(N, n)) + 1j * rng.normal(size=(N, n))
    lam, ms = _product._lambda(s, L, n_theta)[:, lmin**2 :], _lm_m(lmin, L)
    K = L + 1 - lmin
    exact = N * n_theta * n <= LD_BUDGET
    ref, S = _theta_contract(a, lam, ms, L, exact)
    ref, S = ref.reshape(N, -1), S.reshape(N, -1)
    if not exact:
        rows = _sample_rows(N, (K11_CTAS,))
        rr, rS = _theta_contract(a[rows], lam, ms, L, True)
        rr, rS = rr.reshape(rows.size, -1), rS.reshape(rows.size, -1)
    worst = 0.0
    long = None
    for N_run in K11_TIMES:
        got = _theta_synth_run(tb, dev, a[:N_run])
        worst = max(worst, _check_rows(got, ref[:N_run], S[:N_run], K, f"theta_synth {case} N={N_run}", ref_err=0.0 if exact else _ref_err(K)))
        if not exact:
            sel = rows < N_run
            worst = max(worst, check_close(got[rows[sel]], rr[sel], rS[sel], K, f"theta_synth {case} N={N_run} sampled rows"))
        if long is None:
            long = got
        else:
            assert np.array_equal(got.view(np.int64), long[:N_run].view(np.int64)), f"theta_synth {case}: rows differ between launches"
    for r in (1, 2, 3, N - 1):
        assert np.array_equal(_theta_synth_run(tb, dev, a[r : r + 1])[0].view(np.int64), long[r].view(np.int64)), (case, r)
    _note("theta_synth_kernel<9>", worst)


def _theta_quad_run(tb, dev, P, cfg=None):
    import ctypes

    torch = _torch()
    lib = _lib.load()
    N = P.shape[0]
    cfg = np.ascontiguousarray(tb.cfg if cfg is None else cfg, dtype=np.int32)
    d = _upload_rows(P.reshape(N, -1), GUARD)
    before = d.cpu().numpy()
    out = _poisoned((N + GUARD, 2 * tb.n_out))
    _lib.check(lib.scrib200_theta_quad(_lib.ptr(d), N, _lib.ptr(dev["tiles"]), dev["tiles"].shape[0], _lib.ptr(dev["wtfrag"]),
                                       dev["wtfrag"].shape[1], cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(out), _lib.stream_ptr()),
               "theta_quad")
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    check_guard(o, N, f"theta_quad N={N} output")
    assert np.array_equal(d.cpu().numpy().view(np.int64), before.view(np.int64)), "theta_quad: input modified"
    return o[:N].view(complex)


def _quad_problem(case, N):
    s, lmin, L, n_theta, n_phi = case
    rng = np.random.default_rng(80 + THETA_CASES.index(case))
    P = rng.normal(size=(N, n_theta, 2 * L + 1)) + 1j * rng.normal(size=(N, n_theta, 2 * L + 1))
    W = _sf.analysis_tables(s, 0, L, n_theta, n_phi)[1][lmin**2 :]
    return P, W, _lm_m(lmin, L)


@gpu
@pytest.mark.parametrize("case", THETA_CASES, ids=[f"s{c[0]}-lmin{c[1]}-L{c[2]}-{c[3]}x{c[4]}" for c in THETA_CASES])
def test_theta_quad_vs_long_double_reference(case):
    """theta_quad on white noise P (not a band-limited field) at 2371, 1, 3, 4 and 5 steps; at L = 32 the output tiles
    nearly fill the kernel's 8 x 21 (165 of 168 at ell_min = 0) and L = 33 is refused."""
    torch = _torch()
    s, lmin, L, n_theta, n_phi = case
    tb = _product.quad_tables(s, lmin, L, n_theta, n_phi)
    assert tb.fits and int(tb.cfg[2]) == -(-n_theta // 8) and tb.n_out == (L + 1) ** 2 - lmin**2
    tiles = [tuple(x) for x in tb.tiles if x[1] <= L]
    if L == 32:
        assert len(tiles) == {0: 165, 2: 164}[lmin] and tb.tiles.shape[0] == 168
        assert not _product.quad_tables(s, lmin, 33, n_theta, n_phi).fits
    dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(tb, k))).cuda() for k in ("tiles", "wtfrag")}
    N = K11_TIMES[0]
    P, W, ms = _quad_problem(case, N)
    SPa = np.abs(P.real) + np.abs(P.imag)
    K = n_theta
    exact = N * n_theta * tb.n_out <= LD_BUDGET
    ref, S = _quadrature(P, SPa, W, ms, L, exact)
    if not exact:
        # long double on the sampled rows (all columns), and on every row for the elements of the first and last tile of
        # every M
        rows = _sample_rows(N, (K11_CTAS,))
        rr, rS = _quadrature(P[rows], SPa[rows], W, ms, L, True)
        cols = []
        for M in range(-L, L + 1):
            l0s = [l0 for Mi, l0 in tiles if Mi - L == M]
            for l0 in (min(l0s), max(l0s)):
                cols += [l * (l + 1) + M - lmin**2 for l in range(l0, min(l0 + 8, L + 1))]
        cols = np.unique(cols)
        cr, cS = _quadrature(P, SPa, W[cols], ms[cols], L, True)
    worst = 0.0
    long = None
    for N_run in K11_TIMES:
        got = _theta_quad_run(tb, dev, P[:N_run])
        worst = max(worst, _check_rows(got, ref[:N_run], S[:N_run], K, f"theta_quad {case} N={N_run}", ref_err=0.0 if exact else _ref_err(K)))
        if not exact:
            sel = rows < N_run
            worst = max(worst, check_close(got[rows[sel]], rr[sel], rS[sel], K, f"theta_quad {case} N={N_run} sampled rows"))
            worst = max(worst, _check_rows(got[:, cols], cr[:N_run], cS[:N_run], K, f"theta_quad {case} N={N_run} first / last tiles"))
        if long is None:
            long = got
        else:
            assert np.array_equal(got.view(np.int64), long[:N_run].view(np.int64)), f"theta_quad {case}: rows differ between launches"
    for r in (1, 2, 3, N - 1):
        assert np.array_equal(_theta_quad_run(tb, dev, P[r : r + 1])[0].view(np.int64), long[r].view(np.int64)), (case, r)
    _note("theta_quad_kernel<21>", worst)


@gpu
def test_theta_quad_negative_control():
    """theta_quad launched with one ring chunk fewer (cfg[2] - 1): the checker rejects the result."""
    torch = _torch()
    case = THETA_CASES[2]
    s, lmin, L, n_theta, n_phi = case
    tb = _product.quad_tables(s, lmin, L, n_theta, n_phi)
    dev = {k: torch.from_numpy(np.ascontiguousarray(getattr(tb, k))).cuda() for k in ("tiles", "wtfrag")}
    P, W, ms = _quad_problem(case, 5)
    ref, S = _quadrature(P, np.abs(P.real) + np.abs(P.imag), W, ms, L, True)
    assert check_close(_theta_quad_run(tb, dev, P), ref, S, n_theta, "unmodified") < 1.0
    cfg = tb.cfg.copy()
    cfg[2] -= 1
    got = _theta_quad_run(tb, dev, P, cfg=cfg)
    with pytest.raises(AssertionError):
        check_close(got, ref, S, n_theta, "one ring chunk fewer")


# ------------------------------------------------------------------------------------------------------- GPU: grid product
@gpu
@pytest.mark.parametrize("n", [1, 255, 256, 257, 1_000_003])
@pytest.mark.parametrize("in_place", [False, True], ids=["out-of-place", "in-place"])
def test_grid_product_vs_long_double_reference(n, in_place):
    """out = a b elementwise (complex), against a long-double product with K = 2, around the 256-thread block and past the
    grid cap (grid-stride loop); in place (out = a) as grid_multiply(fused=False) calls it."""
    torch = _torch()
    lib = _lib.load()
    rng = np.random.default_rng(n)
    a = (rng.normal(size=n) + 1j * rng.normal(size=n)) * np.exp(rng.uniform(-20, 20, size=n))
    b = (rng.normal(size=n) + 1j * rng.normal(size=n)) * np.exp(rng.uniform(-20, 20, size=n))
    da, db = _upload_rows(a[:, None], GUARD), _upload_rows(b[:, None], GUARD)
    b_before = db.cpu().numpy()
    out = da if in_place else _poisoned((n + GUARD, 2))
    _lib.check(lib.scrib200_grid_product(_lib.ptr(da), _lib.ptr(db), _lib.ptr(out), n, _lib.stream_ptr()), "grid_product")
    torch.cuda.synchronize()
    o = out.cpu().numpy()
    check_guard(o, n, f"grid_product n={n} output")
    assert np.array_equal(db.cpu().numpy().view(np.int64), b_before.view(np.int64)), "grid_product: input modified"
    if not in_place:
        assert np.array_equal(da.cpu().numpy()[:n].view(complex)[:, 0], a), "grid_product: input modified"
    ref = a.astype(np.clongdouble) * b.astype(np.clongdouble)
    S = (np.abs(a.real) + np.abs(a.imag)) * (np.abs(b.real) + np.abs(b.imag))
    _note("grid_product_kernel", check_close(o[:n].view(complex), ref[:, None], S[:, None], 2, f"grid_product n={n}"))


# ------------------------------------------------------------------------------------------------------- GPU: dispatch
@gpu
def test_product_dispatch_under_profiler():
    """Which kernel instantiation runs: one representative launch per kernel under torch.profiler.  The profiling runs in a
    child process: a CUPTI session opened here would stay attached to this process and can leave later profiler sessions of
    the suite (other files' dispatch checks) without kernel records."""
    if os.environ.get("SCRIB200_PRODUCT_PROFILER_CHILD") != "1":
        child = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "gpu",
                                f"{__file__}::test_product_dispatch_under_profiler"],
                               cwd=ROOT, env=dict(os.environ, SCRIB200_PRODUCT_PROFILER_CHILD="1"), capture_output=True, text=True)
        assert child.returncode == 0 and "1 passed" in child.stdout, child.stdout + child.stderr
        return
    import ctypes

    torch = _torch()
    from torch.profiler import ProfilerActivity, profile

    lib = _lib.load()
    rng = np.random.default_rng(6)
    launches = []
    case = K9_CASES["alias-q2"][0]
    a1, a2 = _k9_inputs("alias-q2", 9)
    d1, d2 = torch.from_numpy(a1).cuda(), torch.from_numpy(a2).cuda()
    for shape, kname in K9_SHAPES.items():
        tb = _product.product_tables(*case, shape=shape)
        dev = _k9_device_tables(tb)
        out = torch.empty((9, tb.n_out), dtype=torch.complex128, device="cuda")
        launches.append((kname, lambda tb=tb, dev=dev, out=out: _k9_launch(tb, dev, d1, a1.shape[1], d2, a2.shape[1], 9, out)))
    s, lmin, L, n_theta, n_phi = THETA_CASES[2]
    tt = _product.theta_tables(s, lmin, L, n_theta)
    tdev = {k: torch.from_numpy(np.ascontiguousarray(getattr(tt, k))).cuda() for k in ("perm", "ctl", "lamfrag")}
    a = torch.from_numpy(rng.normal(size=(9, (L + 1) ** 2)) + 0j).cuda()
    Fm = torch.empty((9, n_theta, tt.nm), dtype=torch.complex128, device="cuda")
    launches.append(("theta_synth_kernel<9>", lambda: _lib.check(lib.scrib200_theta_synth(
        _lib.ptr(a), a.shape[1], 9, _lib.ptr(tdev["perm"]), _lib.ptr(tdev["ctl"]), tt.n_ctl, _lib.ptr(tdev["lamfrag"]),
        tdev["lamfrag"].shape[1], tt.cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(Fm), _lib.stream_ptr()), "theta_synth")))
    tq = _product.quad_tables(s, lmin, L, n_theta, n_phi)
    qdev = {k: torch.from_numpy(np.ascontiguousarray(getattr(tq, k))).cuda() for k in ("tiles", "wtfrag")}
    q = torch.empty((9, tq.n_out), dtype=torch.complex128, device="cuda")
    launches.append(("theta_quad_kernel<21>", lambda: _lib.check(lib.scrib200_theta_quad(
        _lib.ptr(Fm), 9, _lib.ptr(qdev["tiles"]), qdev["tiles"].shape[0], _lib.ptr(qdev["wtfrag"]), qdev["wtfrag"].shape[1],
        tq.cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(q), _lib.stream_ptr()), "theta_quad")))
    g = torch.empty(1000, dtype=torch.complex128, device="cuda")
    launches.append(("grid_product_kernel", lambda: _lib.check(lib.scrib200_grid_product(_lib.ptr(Fm), _lib.ptr(Fm), _lib.ptr(g), 1000,
                                                                                         _lib.stream_ptr()), "grid_product")))
    for kname, fn in launches:
        fn()                                                # warm: module loaded, attributes set
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name.replace(" ", "") for e in prof.events() if e.device_type.name == "CUDA"]
        ours = [x for x in names if "scrib200::" in x]
        assert len(ours) == 1 and kname in ours[0], (kname, names)
