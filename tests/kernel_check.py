"""The elementwise checker of the kernel tests (test_gpu_swsh_kernels.py, test_gpu_product_kernels.py): a kernel's output
against a plain high-precision reference of the same operation, with poisoned output buffers and guard rows.

A valid output must be finite and within |out - ref| <= gamma(K) S elementwise, where S is the same contraction taken over
absolute values and K the length of the longest chain of roundings that feeds one output; a guard must come back bit for
bit.  Test infrastructure only."""
import math

import numpy as np

from scri_b200 import _sf

U = 2.0**-53
# gamma = 16 K u, K = the length of the longest chain of roundings that feeds one output: the number of complex terms of
# the synthesis sum, n_theta + n_phi for the analysis (a ring's phi-DFT, then the quadrature over the rings), and for the
# table (ell_max + 1)(ell_max + 2) / 2 (`_table_K`: the upward recurrence in l is neutrally stable at the poles, so an error
# made at step k has grown (l - k)-fold by step l).  Worst-case analysis gives (2K + 2) u for the folded real GEMM with
# its epilogue, (3K + 8) u for the three-multiplication product and about 3 (K + 4) u for the two analysis stages with
# complex rounding, all measured against the absolute-value contraction S: 16 K u covers each for every K >= 1 without a
# per-kernel constant, and is still some 1e12 times smaller than the change a dropped mode or a shifted column makes.
GAMMA_PER_TERM = 16


def gamma(K):
    return GAMMA_PER_TERM * K * U


def _real_view(x):
    x = np.asarray(x)
    if np.iscomplexobj(x):
        return np.stack([x.real, x.imag], axis=-1).reshape(x.shape[:-1] + (2 * x.shape[-1],))
    return x


def check_close(out, ref, S, K, what, ref_err=0.0):
    """|out - ref| <= (gamma(K) + ref_err) * S elementwise, and out finite.

    out, ref: arrays of one shape (complex ones are compared part by part); S: the same contraction over absolute values,
    either per real part ([..., 2 n]) or per complex element ([..., n], applied to both parts).  `ref_err` is the
    worst-case relative error of a float64 reference (0 for a long-double one).  Returns max |out - ref| / (gamma S)."""
    o = _real_view(out).astype(np.float64)
    r = _real_view(ref)
    S = np.asarray(S, dtype=np.float64)
    if np.iscomplexobj(out) and S.shape == np.shape(out):
        S = np.repeat(S, 2, axis=-1)
    assert o.shape == r.shape == S.shape, (what, o.shape, r.shape, S.shape)
    err = np.abs(o.astype(r.dtype) - r).astype(np.float64)
    bound = (gamma(K) + ref_err) * S
    ok = np.isfinite(o) & (err <= bound)
    if not ok.all():
        bad = np.argwhere(~ok.reshape(ok.shape[0], -1) if ok.ndim > 1 else ~ok[:, None])
        rows, cols = np.unique(bad[:, 0]), np.unique(bad[:, 1])
        i = tuple(np.argwhere(~ok)[0])
        raise AssertionError(
            f"{what}: {bad.shape[0]} of {ok.size} elements outside |out - ref| <= gamma S (gamma = {gamma(K):.3g}); "
            f"{np.count_nonzero(~np.isfinite(o))} not finite; rows {rows[:12].tolist()}{' ...' if rows.size > 12 else ''} "
            f"(of {rows.size}), real columns {cols[:12].tolist()}{' ...' if cols.size > 12 else ''} (of {cols.size}); "
            f"first at {i}: out {o[i]!r} ref {float(r[i])!r} bound {bound[i]:.3g}")
    with np.errstate(invalid="ignore", divide="ignore"):
        ratio = np.where(S > 0, err / (gamma(K) * S), 0.0)
    return float(ratio.max()) if ratio.size else 0.0


POISON = 0x7FF8DEADBEEF0BAD   # a quiet NaN with a payload no arithmetic produces


def check_guard(buf, n_valid, what):
    """Rows n_valid.. of a poisoned float64 buffer still hold the poison pattern, bit for bit."""
    g = np.ascontiguousarray(buf[n_valid:]).view(np.int64)
    assert (g == POISON).all(), f"{what}: {np.count_nonzero(g != POISON)} guard words overwritten"


# ------------------------------------------------------------------------------------------------------- GPU helpers
def _torch():
    import torch

    return torch


def _poisoned(shape):
    torch = _torch()
    t = torch.empty(shape, dtype=torch.float64, device="cuda")
    t.view(torch.int64).fill_(POISON)
    return t


def _upload_rows(host, guard):
    """Device float64 copy of a complex [N, n] array with `guard` poisoned rows after it."""
    torch = _torch()
    h = _real_view(host)
    d = _poisoned((h.shape[0] + guard, h.shape[1]))
    d[: h.shape[0]] = torch.from_numpy(np.ascontiguousarray(h)).cuda()
    return d


GUARD = 3
WORST = {}   # largest |out - ref| / (gamma S) per kernel, printed by each case (pytest -s)


def _note(kernel, ratio):
    WORST[kernel] = max(WORST.get(kernel, 0.0), ratio)
    print(f"\n[{kernel}] max |out - ref| / (gamma S) = {ratio:.3g} (worst so far {WORST[kernel]:.3g})")


# ---------------------------------------------------------------------------------------- bound of a Wigner-d table
def _table_scale(R, s, ell_min, ell_max, Lt):
    """Elementwise scale of sY_lm(R_g) = c_l PhA PhB P^l for the table bound: c_l |Ra|^|mp+m| |Rb|^|m-mp| max_{l'<=l} |P^l'|,
    m = -s, with the phase magnitude floored at the smallest normal number (below it rounding is absolute, not relative)."""
    R = np.asarray(R, dtype=float)
    Ra, Rb = R[:, 0] + 1j * R[:, 3], R[:, 2] + 1j * R[:, 1]
    cosb = (np.abs(Ra) ** 2) - (np.abs(Rb) ** 2)
    seed, rec = _sf.wigner_tables(Lt)
    m = -s
    out = np.zeros((R.shape[0], _sf.LM_total_size(ell_min, ell_max)))
    for mp in range(-ell_max, ell_max + 1):
        l0 = max(abs(mp), abs(m))
        if l0 > ell_max:
            continue
        mag = np.maximum(np.abs(Ra) ** abs(mp + m) * np.abs(Rb) ** abs(m - mp), np.finfo(float).tiny)
        Pl, Pm1 = np.full(R.shape[0], seed[mp + Lt, m + Lt]), np.zeros(R.shape[0])
        run = np.abs(Pl)
        for ell in range(l0, ell_max + 1):
            run = np.maximum(run, np.abs(Pl))
            if ell >= ell_min:
                out[:, _sf.LM_index(ell, mp, ell_min)] = math.sqrt((2 * ell + 1) / (4 * math.pi)) * mag * run
            if ell < ell_max:
                ca, cb, cc = rec[ell, mp + Lt, m + Lt]
                Pl, Pm1 = (ca * cosb - cb) * Pl - cc * Pm1, Pl
    return out


def _table_K(ell_max):
    return (ell_max + 1) * (ell_max + 2) // 2
