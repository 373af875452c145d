"""Time-domain inner products: the spline integration weights (host), `mode_calculations.inner_product`,
`WaveformModes.inner_product`, `mode_calculations.inner_product_matrix` and the two kernels behind them (csrc/inner.cu).

No golden vector covers these functions, so they are pinned by scipy (the weights against
InterpolatedUnivariateSpline.integral, which is what quaternion.calculus.spline_definite_integral calls) and by the oracle's
restatement of the reference flow (oracle/inner_product_ref.py: inner_product, waveform_inner_product).

Bars.  Against the oracle: |out - ref| <= 1e-12 S, S = sum_i |w_i| sum_m |a||b| (the same integral over absolute values, so
cancellation neither hides nor inflates an error).  Kernel cases through the C ABI: against a long-double contraction with
the same weights at gamma S, gamma = 16 K 2^-53 (K = terms per output), as in test_gpu_swsh_kernels.py; outputs start as a
NaN pattern followed by guard elements that must come back bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.interpolate import InterpolatedUnivariateSpline

import scri_b200 as sb
from oracle import inner_product_ref as IP
from oracle import scri_ref as R
from scri_b200 import _lib, ops
from scri_b200 import mode_calculations as mc
from scri_b200.flux import intersection

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

U = 2.0**-53
ORACLE_BAR = 1e-12
WEIGHT_BAR = 1e-13        # measured worst case over the cases below: 3.4e-15 of sum |w_ref|
POISON = 0x7FF8DEADBEEF0BAD
GUARD = 8


def _sdi(f, t, t1=None, t2=None, axis=None):
    return IP._refshim_calculus().spline_definite_integral(f, t, t1=t1, t2=t2, axis=axis)


def _axis(N, kind, seed=0):
    if kind == "uniform":
        return np.linspace(-1.0, 3.0, N)
    t = np.sort(np.random.default_rng(seed).uniform(-1.0, 3.0, N))
    t[0], t[-1] = -1.0, 3.0
    return t


def _bounds(t):
    N = t.size
    k = t[min(2, N - 1)]
    return [
        (None, None),
        (t[0] + 0.3 * (t[1] - t[0]), t[-1] - 0.7 * (t[-1] - t[-2])),       # interior, off the samples
        (t[1], t[-2]),                                                      # on samples (on knots for N > 5)
        (k, k),                                                             # t1 == t2
        (2.5, -0.5),                                                        # t1 > t2
        (-5.0, 1.0), (0.5, 9.0), (-5.0, 9.0),                               # one or both outside
        (-9.0, -5.0), (5.0, 9.0),                                           # both outside on one side
    ]


# ----------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("kind", ["uniform", "random"])
@pytest.mark.parametrize("N", [4, 5, 7, 33, 1000])
def test_weights_match_scipy(N, kind):
    t = _axis(N, kind, seed=N)
    eye = np.eye(N)
    for t1, t2 in _bounds(t):
        w = ops.spline_integral_weights(t, t1, t2)
        a = t[0] if t1 is None else t1
        b = t[-1] if t2 is None else t2
        ref = np.array([InterpolatedUnivariateSpline(t, eye[j], k=3).integral(a, b) for j in range(N)])
        assert np.abs(w - ref).max() <= WEIGHT_BAR * np.abs(ref).sum(), (N, kind, t1, t2)


def test_weights_need_four_samples():
    with pytest.raises(ValueError):
        ops.spline_integral_weights(np.arange(3.0))


@pytest.mark.parametrize("N", [4, 9, 500])
def test_weights_linearity(N):
    rng = np.random.default_rng(N)
    t = _axis(N, "random", seed=N + 1)
    f = rng.normal(size=(N, 6)) + 1j * rng.normal(size=(N, 6))
    for t1, t2 in [(None, None), (-0.3, 2.2), (2.0, -3.0)]:
        w = ops.spline_integral_weights(t, t1, t2)
        ref = _sdi(f, t, t1, t2, axis=0)
        S = np.abs(w) @ np.abs(f)
        assert (np.abs(w @ f - ref) <= 1e-12 * S).all()


def _wm(t, data, ell_min=2, ell_max=8, dataType=sb.h):
    return sb.WaveformModes(t=t, data=data, ell_min=ell_min, ell_max=ell_max, frameType=sb.Inertial, dataType=dataType,
                            r_is_scaled_out=True, m_is_scaled_out=True)


def _random_modes(t, ell_min, ell_max, seed):
    rng = np.random.default_rng(seed)
    n = ell_max * (ell_max + 2) - ell_min**2 + 1
    return rng.normal(size=(t.size, n)) + 1j * rng.normal(size=(t.size, n))


def test_argument_errors():
    """Each check raises before any device work, with the type and message of flux.matrix_expectation_value's checks."""
    t = np.linspace(0.0, 1.0, 11)
    a = _wm(t, _random_modes(t, 2, 8, 0))
    cases = [
        (_wm(t, _random_modes(t, 2, 8, 1), dataType=sb.psi3), {}, "Spin weights must match in inner_product"),
        (_wm(t, _random_modes(t, 2, 6, 2), ell_max=6), {},
         "ell_min and ell_max must match in inner_product (use allow_LM_differ=True to override)"),
        (_wm(t, _random_modes(t, 9, 10, 3), ell_min=9, ell_max=10), dict(allow_LM_differ=True),
         "Intersection of (ell,m) modes is empty.  Assuming this is not desired."),
        (_wm(t + 0.01, _random_modes(t, 2, 8, 4)), {},
         "Time samples must match in inner_product (use allow_times_differ=True to override)"),
    ]
    for b, kw, msg in cases:
        with pytest.raises(ValueError) as e:
            a.inner_product(b, **kw)
        assert str(e.value) == msg
        with pytest.raises(ValueError) as e:
            IP.waveform_inner_product(R.Modes(t=a.t, data=a.data), R.Modes(t=b.t, data=b.data, ell_min=b.ell_min, ell_max=b.ell_max,
                                                                         dataType=b.dataType), **kw)
        assert str(e.value) == msg


def test_no_cpu_fallback():
    """Without a CUDA device the three operators raise Scrib200Error; on a machine with a device this test runs again in a
    child process that is shown none."""
    import torch

    if torch.cuda.is_available():
        child = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{__file__}::test_no_cpu_fallback"],
                               cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
        assert child.returncode == 0 and "1 passed" in child.stdout, child.stdout + child.stderr
        return
    t = np.linspace(0.0, 1.0, 11)
    d = _random_modes(t, 2, 8, 0)
    w = _wm(t, d)
    with pytest.raises(_lib.Scrib200Error):
        mc.inner_product(t, d, d)
    with pytest.raises(_lib.Scrib200Error):
        w.inner_product(w)
    with pytest.raises(_lib.Scrib200Error):
        mc.inner_product_matrix(t, d[None], d[None])


# ----------------------------------------------------------------------------------------------------------- GPU
def _oracle_close(out, ref, S, what):
    err = np.abs(np.asarray(out) - np.asarray(ref))
    assert np.all(np.isfinite(out)), what
    assert (err <= ORACLE_BAR * np.asarray(S)).all(), (what, float(np.max(err / np.maximum(S, 1e-300))))
    return float(np.max(err / np.maximum(ORACLE_BAR * np.asarray(S), 1e-300)))


@gpu
def test_mode_calculations_inner_product_layouts():
    import torch

    rng = np.random.default_rng(5)
    N, n = 301, 7
    t = _axis(N, "random", seed=3)
    w = ops.spline_integral_weights(t)
    worst = 0.0
    for is_complex in (True, False):
        mk = (lambda *s: rng.normal(size=s) + 1j * rng.normal(size=s)) if is_complex else (lambda *s: rng.normal(size=s))
        for conj in (False, True):
            a, b = mk(N, n), mk(N, n)
            ref = IP.inner_product(t, a, b, axis=0, apply_conjugate=conj)
            S = np.abs(w) @ (np.abs(a) * np.abs(b))
            for axis in (0, None):
                out = mc.inner_product(t, a, b, axis=axis, apply_conjugate=conj)
                assert out.shape == ref.shape and out.dtype == ref.dtype, (out.shape, out.dtype, ref.dtype)
                worst = max(worst, _oracle_close(out, ref, S, f"[N, n] axis={axis}"))
            aT, bT = np.ascontiguousarray(a.T), np.ascontiguousarray(b.T)
            out = mc.inner_product(t, aT, bT, axis=1, apply_conjugate=conj)
            worst = max(worst, _oracle_close(out, IP.inner_product(t, aT, bT, axis=1, apply_conjugate=conj), S, "[n, N] axis=1"))
            outd = mc.inner_product(t, torch.from_numpy(aT).cuda(), torch.from_numpy(bT).cuda(), axis=1, apply_conjugate=conj)
            assert outd.is_cuda and np.array_equal(outd.cpu().numpy(), out)
            a1, b1 = a[:, 0].copy(), b[:, 0].copy()
            out = mc.inner_product(t, a1, b1, apply_conjugate=conj)
            ref1 = IP.inner_product(t, a1, b1, apply_conjugate=conj)
            assert out.shape == ref1.shape == ()
            worst = max(worst, _oracle_close(out, ref1, S[0], "1-D"))
    print(f"mode_calculations.inner_product: largest error / bar {worst:.3g}")


def _pair_S(w, A, B):
    return float(np.abs(w) @ np.sum(np.abs(A) * np.abs(B), axis=1))


@gpu
def test_waveform_inner_product_fake_precessing():
    a = sb.sample_waveforms.fake_precessing_waveform(t_0=-20.0, t_1=1980.0, dt=0.1, ell_max=8)
    assert abs(a.n_times - 20000) <= 1
    b = a.copy()
    b.data = a.data * np.exp(0.3j) + 0.1 * np.roll(a.data, 3, axis=1)
    Ra, Rb = (R.Modes(t=x.t, data=x.data, ell_min=x.ell_min, ell_max=x.ell_max) for x in (a, b))
    worst = 0.0
    for t1, t2 in [(None, None), (100.0, 1500.5), (-500.0, 3000.0), (1700.0, 200.0)]:
        out = a.inner_product(b, t1=t1, t2=t2)
        ref = IP.waveform_inner_product(Ra, Rb, t1=t1, t2=t2)
        S = _pair_S(ops.spline_integral_weights(a.t, t1, t2), a.data, b.data)
        worst = max(worst, _oracle_close(out, ref, S, f"<a,b> over ({t1}, {t2})"))
        back = b.inner_product(a, t1=t1, t2=t2)
        assert abs(back - np.conj(out)) <= ORACLE_BAR * S
    aa = a.inner_product(a)
    S = _pair_S(ops.spline_integral_weights(a.t), a.data, a.data)
    assert abs(aa.imag) <= ORACLE_BAR * S and aa.real >= 0
    assert abs(aa.real - _sdi(ops.norm(a.data), a.t)) <= ORACLE_BAR * S
    print(f"WaveformModes.inner_product (fake precessing): largest error / bar {worst:.3g}")


@gpu
def test_waveform_inner_product_random_modes_ell_and_time_clipping():
    t = np.linspace(0.0, 50.0, 1201)
    a = _wm(t, _random_modes(t, 2, 8, 10))
    b = _wm(t, _random_modes(t, 3, 6, 11), ell_min=3, ell_max=6)
    Ra = R.Modes(t=a.t, data=a.data)
    Rb = R.Modes(t=b.t, data=b.data, ell_min=3, ell_max=6)
    out = a.inner_product(b, allow_LM_differ=True)
    ref = IP.waveform_inner_product(Ra, Rb, allow_LM_differ=True)
    A = a.data[:, 9 - 4 : 6 * 8 + 1 - 4]
    S = _pair_S(ops.spline_integral_weights(t), A, b.data)
    _oracle_close(out, ref, S, "allow_LM_differ")
    assert abs(b.inner_product(a, allow_LM_differ=True) - np.conj(out)) <= ORACLE_BAR * S
    # two offset non-uniform axes
    rng = np.random.default_rng(12)
    t1 = np.sort(rng.uniform(0.0, 60.0, 1500))
    t2 = np.sort(rng.uniform(5.0, 70.0, 1400))
    f = lambda tt, seed: np.exp(1j * np.outer(tt, np.random.default_rng(seed).uniform(0.05, 0.4, 77))) * np.random.default_rng(seed + 1).normal(size=77)
    a, b = _wm(t1, f(t1, 20)), _wm(t2, f(t2, 20) * 1.1)
    out = a.inner_product(b, allow_times_differ=True)
    ref = IP.waveform_inner_product(R.Modes(t=a.t, data=a.data), R.Modes(t=b.t, data=b.data), allow_times_differ=True,
                                   intersection=intersection)
    tc = intersection(t1, t2)
    Ai, Bi = a.interpolate(tc).data, b.interpolate(tc).data
    _oracle_close(out, ref, _pair_S(ops.spline_integral_weights(tc), Ai, Bi), "allow_times_differ")
    with_both = a[:, 3:7].inner_product(b, allow_times_differ=True, allow_LM_differ=True)
    ref2 = IP.waveform_inner_product(R.Modes(t=a.t, data=a[:, 3:7].data, ell_min=3, ell_max=6), R.Modes(t=b.t, data=b.data),
                                    allow_times_differ=True, allow_LM_differ=True, intersection=intersection)
    _oracle_close(with_both, ref2, _pair_S(ops.spline_integral_weights(tc), Ai[:, 5:45], Bi[:, 5:45]), "both")


# ------------------------------------------------------------------------------------------ kernels through the C ABI
def _poisoned(torch, n_complex):
    buf = torch.empty(2 * (n_complex + GUARD), dtype=torch.float64, device="cuda")
    buf.view(torch.int64).fill_(POISON)
    return buf


def _check_guard(buf, n_complex, what):
    g = buf.cpu().numpy()[2 * n_complex:].view(np.int64)
    assert (g == POISON).all(), f"{what}: guard overwritten"


def _ld_reference(A, B, w, conj, per_column):
    """Long-double contraction with the same weights, and the absolute-value contraction S."""
    Al, Bl = A.astype(np.clongdouble), B.astype(np.clongdouble)
    P = (np.conj(Al) if conj else Al) * Bl * w.astype(np.longdouble)[:, None]
    S = (np.abs(w)[:, None] * np.abs(A) * np.abs(B))
    if per_column:
        return P.sum(axis=0), S.sum(axis=0)
    return P.sum(), S.sum()


def _run_stream(torch, lib, a, b, w, n, a0=0, b0=0, conj=1, per_column=0):
    N = a.shape[0]
    nout = n if per_column else 1
    out = _poisoned(torch, nout)
    ws = torch.empty(max(16, lib.scrib200_inner_product_workspace_bytes(N, n, 1)), dtype=torch.uint8, device="cuda")
    _lib.check(lib.scrib200_inner_product(_lib.ptr(a), a.shape[1], a0, 0, _lib.ptr(b), b.shape[1], b0, 0, N, n, 1, _lib.ptr(w),
                                          conj, per_column, _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "inner_product")
    torch.cuda.synchronize()
    _check_guard(out, nout, "inner_product")
    return out[: 2 * nout].cpu().numpy().view(np.complex128)


def _stream_case(torch, lib, N, n, pitch_a, pitch_b, a0, b0, seed):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(N, pitch_a)) + 1j * rng.normal(size=(N, pitch_a))
    B = rng.normal(size=(N, pitch_b)) + 1j * rng.normal(size=(N, pitch_b))
    t = np.cumsum(rng.uniform(0.5, 1.5, N))
    w = ops.spline_integral_weights(t, t[0] + 0.1, t[-1] - 0.2)
    a, b, wd = (torch.from_numpy(x).cuda() for x in (A, B, w))
    worst = 0.0
    Aw, Bw = A[:, a0 : a0 + n], B[:, b0 : b0 + n]
    for conj in (1, 0):
        for per_column in (0, 1):
            out = _run_stream(torch, lib, a, b, wd, n, a0, b0, conj, per_column)
            again = _run_stream(torch, lib, a, b, wd, n, a0, b0, conj, per_column)
            assert np.array_equal(out.view(np.int64), again.view(np.int64)), "two launches differ"
            ref, S = _ld_reference(Aw, Bw, w, conj, per_column)
            K = N if per_column else N * n
            ref_parts = np.stack([np.real(ref), np.imag(ref)], axis=-1)
            out_parts = np.stack([out.real, out.imag], axis=-1).reshape(ref_parts.shape)
            err = np.abs(out_parts.astype(np.longdouble) - ref_parts).astype(float)
            bound = 16 * K * U * np.asarray(S, dtype=float)[..., None]
            assert np.isfinite(out).all() and (err <= bound).all(), (N, n, conj, per_column, float((err / bound).max()))
            worst = max(worst, float((err / np.maximum(bound, 1e-300)).max()))
    return worst


@gpu
@pytest.mark.parametrize("N", [4, 5, 31, 32, 33, 255, 256, 257])
def test_streaming_kernel_lengths(N):
    import torch

    lib = _lib.load()
    worst = _stream_case(torch, lib, N, 5, 5, 5, 0, 0, seed=N)
    print(f"inner_product N={N}: largest error / (gamma S) {worst:.3g}")


@gpu
@pytest.mark.parametrize("n", [1, 5, 77, 285, 1089])
def test_streaming_kernel_widths_and_windows(n):
    import torch

    lib = _lib.load()
    worst = _stream_case(torch, lib, 1000, n, n, n, 0, 0, seed=n)
    worst = max(worst, _stream_case(torch, lib, 613, n, n + 9, n + 3, 7, 2, seed=n + 1))      # clipped views: pitch != window
    print(f"inner_product n={n}: largest error / (gamma S) {worst:.3g}")


@gpu
def test_streaming_kernel_million_steps():
    import torch

    lib = _lib.load()
    worst = _stream_case(torch, lib, 1_000_000, 3, 3, 3, 0, 0, seed=99)
    print(f"inner_product N=1e6: largest error / (gamma S) {worst:.3g}")


def _ld_matrix(A, B, w):
    Al = np.conj(A.reshape(A.shape[0], -1).astype(np.clongdouble)) * np.repeat(w.astype(np.longdouble), A.shape[2])[None, :]
    G = Al @ B.reshape(B.shape[0], -1).astype(np.clongdouble).T
    S = (np.abs(A.reshape(A.shape[0], -1)) * np.repeat(np.abs(w), A.shape[2])[None, :]) @ np.abs(B.reshape(B.shape[0], -1)).T
    return G, S


def _run_matrix(torch, lib, Ad, Bd, wd):
    P, N, n = Ad.shape
    Q = Bd.shape[0]
    G = _poisoned(torch, P * Q)
    ws = torch.empty(max(16, lib.scrib200_inner_product_matrix_workspace_bytes(P, Q, N, n)), dtype=torch.uint8, device="cuda")
    _lib.check(lib.scrib200_inner_product_matrix(_lib.ptr(Ad), P, N * n, _lib.ptr(Bd), Q, N * n, N, n, _lib.ptr(wd), _lib.ptr(G),
                                                 _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "inner_product_matrix")
    torch.cuda.synchronize()
    _check_guard(G, P * Q, "inner_product_matrix")
    return G[: 2 * P * Q].cpu().numpy().view(np.complex128).reshape(P, Q)


@gpu
@pytest.mark.parametrize("P,Q", [(1, 1), (1, 9), (130, 1), (2, 2), (7, 8), (8, 9), (9, 64), (64, 65), (65, 130), (130, 7)])
def test_matrix_kernel(P, Q):
    import torch

    lib = _lib.load()
    rng = np.random.default_rng(P * 1000 + Q)
    N, n = 203, 13                                # K = 2639: ragged against the 8-term stages and the K split
    t = np.cumsum(rng.uniform(0.5, 1.5, N))
    w = ops.spline_integral_weights(t, t[3], t[-1] + 5.0)
    A = rng.normal(size=(P, N, n)) + 1j * rng.normal(size=(P, N, n))
    B = rng.normal(size=(Q, N, n)) + 1j * rng.normal(size=(Q, N, n))
    Ad, Bd, wd = (torch.from_numpy(x).cuda() for x in (A, B, w))
    G = _run_matrix(torch, lib, Ad, Bd, wd)
    assert np.array_equal(G.view(np.int64), _run_matrix(torch, lib, Ad, Bd, wd).view(np.int64)), "two launches differ"
    ref, S = _ld_matrix(A, B, w)
    bound = 16 * N * n * U * S
    err = np.maximum(np.abs(G.real - np.real(ref).astype(float)), np.abs(G.imag - np.imag(ref).astype(float)))
    assert np.isfinite(G).all() and (err <= bound).all(), float((err / bound).max())
    # against the pairwise streaming kernel
    for p, q in {(0, 0), (P - 1, Q - 1), (P // 2, Q // 3)}:
        pair = ops.inner_product(Ad[p], Bd[q], wd).cpu().numpy()
        assert abs(G[p, q] - pair) <= 1e-12 * S[p, q]
    print(f"inner_product_matrix P={P} Q={Q}: largest error / (gamma S) {float((err / bound).max()):.3g}")


@gpu
def test_matrix_kernel_self_is_hermitian():
    import torch

    rng = np.random.default_rng(3)
    P, N, n = 65, 150, 21
    t = np.sort(rng.uniform(0.0, 10.0, N))
    A = torch.from_numpy(rng.normal(size=(P, N, n)) + 1j * rng.normal(size=(P, N, n))).cuda()
    G = mc.inner_product_matrix(t, A, A).cpu().numpy()
    w = ops.spline_integral_weights(t)
    _, S = _ld_matrix(A.cpu().numpy(), A.cpu().numpy(), w)
    assert (np.abs(G - G.conj().T) <= ORACLE_BAR * S).all()
    assert (np.abs(np.diag(G).imag) <= ORACLE_BAR * np.diag(S)).all() and (np.diag(G).real >= 0).all()


@gpu
def test_matrix_dispatch_under_profiler():
    """The DMMA kernel runs for P, Q > 1 and the streaming kernel for a single row or column of G.  The profiling runs in a
    child process: a CUPTI session opened here would stay attached to this process and can leave later profiler sessions
    of the suite (other files' dispatch checks) without kernel records."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    if os.environ.get("SCRIB200_INNER_PROFILER_CHILD") != "1":
        child = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "gpu",
                                f"{__file__}::test_matrix_dispatch_under_profiler"],
                               cwd=ROOT, env=dict(os.environ, SCRIB200_INNER_PROFILER_CHILD="1"), capture_output=True, text=True)
        assert child.returncode == 0 and "1 passed" in child.stdout, child.stdout + child.stderr
        return
    rng = np.random.default_rng(4)
    N, n = 64, 9
    t = np.linspace(0.0, 1.0, N)
    mk = lambda P: torch.from_numpy(rng.normal(size=(P, N, n)) + 1j * rng.normal(size=(P, N, n))).cuda()
    for P, Q, expect, absent in [(5, 6, "inner_product_dmma_kernel", "inner_product_kernel"),
                                 (1, 6, "inner_product_kernel", "inner_product_dmma_kernel"),
                                 (6, 1, "inner_product_kernel", "inner_product_dmma_kernel")]:
        A, B = mk(P), mk(Q)
        mc.inner_product_matrix(t, A, B)          # warm: weights cached, module loaded
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            mc.inner_product_matrix(t, A, B)
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type.name == "CUDA"]
        assert any(expect in x for x in names), (P, Q, names)
        assert not any(absent in x for x in names), (P, Q, names)


@gpu
def test_matrix_of_a_transformed_batch():
    """G of one batch out of parallel.transform_batch equals WaveformModes.inner_product of the same pair."""
    from scri_b200 import parallel
    from scri_b200 import plan as Pl

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from scri_inputs import real_supertranslation, smooth_modes

    Bn, N = 6, 400
    t = np.linspace(0.0, 60.0, N)
    batch = np.stack([smooth_modes(n_times=N, t0=0.0, t1=60.0, seed=300 + b)[1] for b in range(Bn)])
    plan = Pl.TransformPlan(2, 8, sb.h, supertranslation=real_supertranslation(3), frame_rotation=[1.0, 2.0, 3.0, 4.0])
    up, out = parallel.transform_batch(plan, ops.to_device(t), ops.to_device(batch))
    G = mc.inner_product_matrix(up, out, out).cpu().numpy()
    u = up.cpu().numpy()
    host = out.cpu().numpy()
    w = ops.spline_integral_weights(u)
    for p, q in [(0, 0), (1, 4), (5, 2)]:
        wp, wq = _wm(u, host[p].copy()), _wm(u, host[q].copy())
        S = _pair_S(w, host[p], host[q])
        assert abs(G[p, q] - wp.inner_product(wq)) <= ORACLE_BAR * S
