"""<L>, <LL>, dominant eigenvector, angular velocity, corotating frame (mirrors scri/mode_calculations.py).

The per-time-step reductions run on the GPU (csrc/modes.cu).  The serial pieces the reference delegates to
numpy-quaternion - integrating the angular velocity (mode_calculations.py:467) and `minimal_rotation`
(rotations.py:39) - stay on the host with scipy, as SURVEY.md 8(a18)/8(f2) schedules them.
"""
import numpy as np

from . import _quaternion as Q
from . import _lib, ops


def LdtVector(W):
    r"""<L d/dt>^a = sum conj(f)^{l,m'} <l,m'|L_a|l,m> (df/dt)^{l,m}   (scri/mode_calculations.py:46-57)"""
    _, Ldt = ops.ll_ldt(W.data, W.data_dot, W.ell_min, W.ell_max)
    return Ldt


def LVector(W):
    r"""<L>^a = sum conj(f)^{l,m'} <l,m'|L_a|l,m> f^{l,m}   (scri/mode_calculations.py:92-103)"""
    return ops.l_vector(W.data, W.data, W.ell_min, W.ell_max)


def LLMatrix(W):
    r"""<LL>^{ab} = Re sum conj(f)^{l,m'} <l,m'|L_a L_b|l,m> f^{l,m}   (scri/mode_calculations.py:298-313)"""
    LL, _ = ops.ll_ldt(W.data, None, W.ell_min, W.ell_max)
    return LL


def LLComparisonMatrix(W1, W2):
    r"""<LL>^{ab} = sum conj(f)^{l,m'} <l,m'|L_a L_b|l,m> g^{l,m} between two waveforms, complex
    (scri/mode_calculations.py:195-206)"""
    return ops.ll_comparison(W1.data, W2.data, W1.ell_min, W1.ell_max)


def LLDominantEigenvector(W, RoughDirection=np.array([0.0, 0.0, 1.0]), RoughDirectionIndex=0):
    """Principal axis of <LL>, sign-continuous in time (scri/mode_calculations.py:366-399)."""
    torch_data = ops.to_device(W.data, np.complex128)
    LL, _ = ops.ll_ldt(torch_data, None, W.ell_min, W.ell_max)
    dpa = ops.dominant_eigenvector(LL, ops.to_device(np.asarray(RoughDirection, dtype=float)), RoughDirectionIndex)
    return ops.to_host(dpa)


def angular_velocity(W, include_frame_velocity=False):
    """omega = -<LL>^{-1} <L d/dt>   (scri/mode_calculations.py:403-432)"""
    d = ops.to_device(W.data, np.complex128)
    t = ops.to_device(W.t, np.float64)
    ddot = ops.spline_calculus(t, d, "derivative", 1)
    LL, Ldt = ops.ll_ldt(d, ddot, W.ell_min, W.ell_max)
    omega = ops.to_host(ops.solve3(LL, Ldt, scale=-1.0))
    if include_frame_velocity and len(W.frame) == W.n_times:
        from scipy.interpolate import CubicSpline

        Rdot = CubicSpline(W.t, W.frame).derivative()(W.t)
        omega += (2 * Q.qmul(Rdot, Q.qconj(W.frame)))[:, 1:]
    return omega


def integrate_angular_velocity(t, omega, R0=(1.0, 0.0, 0.0, 0.0), tolerance=1e-12):
    """Rotor series with dR/dt = omega R / 2, R(t[0]) = R0, on the samples `t`.

    Stand-in for quaternion.integrate_angular_velocity (scri/mode_calculations.py:467): cubic-spline omega, Dormand-Prince
    8(5,3) with absolute tolerance `tolerance`.  One serial ODE over the whole series - host work by nature - run by the
    native integrator of the library (scrib200_integrate_angular_velocity) instead of scipy's DOP853 with a Python
    right-hand side (1.3 s for 2e4 samples, ~60 000 interpreter round trips): the steps are clipped to the samples, so no
    dense output is needed.
    """
    import ctypes

    from scipy.interpolate import CubicSpline

    t = np.ascontiguousarray(t, dtype=float)
    coef = np.ascontiguousarray(CubicSpline(t, np.asarray(omega, dtype=float)).c)          # [4, n-1, 3]
    R0 = np.ascontiguousarray(R0, dtype=float)
    out = np.empty((t.shape[0], 4))
    if t.shape[0] == 1:
        out[0] = R0
        return out
    lib = _lib.load()
    _lib.check(
        lib.scrib200_integrate_angular_velocity(t.ctypes.data, t.shape[0], coef.ctypes.data, R0.ctypes.data, float(tolerance), 1e-13,
                                                out.ctypes.data, None),
        "integrate_angular_velocity",
    )
    return out


def corotating_frame(W, R0=(1.0, 0.0, 0.0, 0.0), tolerance=1e-12, z_alignment_region=None, return_omega=False):
    """Rotor taking the current mode frame into the corotating frame (scri/mode_calculations.py:435-490)."""
    omega = angular_velocity(W)
    frame = integrate_angular_velocity(W.t, omega, R0=Q.as_float_quat(R0), tolerance=tolerance)
    if z_alignment_region is None:
        correction_rotor = np.array([1.0, 0.0, 0.0, 0.0])
    else:
        initial_time = W.t[0]
        inspiral_time = W.max_norm_time() - initial_time
        t1 = initial_time + z_alignment_region[0] * inspiral_time
        t2 = initial_time + z_alignment_region[1] * inspiral_time
        i1 = np.argmin(np.abs(W.t - t1))
        i2 = np.argmin(np.abs(W.t - t2))
        R = frame[i1:i2]
        i1m = max(0, i1 - 10)
        RoughDirection = omega[i1m + 10]
        LL, _ = ops.ll_ldt(np.ascontiguousarray(W.data[i1:i2]), None, W.ell_min, W.ell_max)
        Vhat = ops.dominant_eigenvector(LL, RoughDirection, 0)
        Vq = np.concatenate([np.zeros((Vhat.shape[0], 1)), Vhat], axis=1)
        Vhat_corot = Q.qmul(Q.qmul(Q.qconj(R), Vq), R)[:, 1:]
        mean = np.mean(Vhat_corot, axis=0)
        mean_q = Q.qnormalized(np.array([0.0, mean[0], mean[1], mean[2]]))
        zq = np.array([0.0, 0.0, 0.0, 1.0])
        correction_rotor = Q.qinverse(Q.qsqrt(-Q.qmul(zq, mean_q)))
    frame = Q.qmul(frame, correction_rotor)
    frame = frame / Q.qabs(frame)[:, None]
    if return_omega:
        return (frame, omega)
    return frame


def minimal_rotation(R, t, iterations=2):
    """Remove rotation about z from the rotor series (quaternion.minimal_rotation; used at scri/rotations.py:39)."""
    from scipy.interpolate import CubicSpline

    R = np.asarray(R, dtype=float)
    zq = np.array([0.0, 0.0, 0.0, 1.0])
    for _ in range(iterations):
        Rdot = CubicSpline(t, R).derivative()(t)
        halfgammadot = Q.qmul(Q.qmul(Rdot, zq), Q.qconj(R))[:, 0]
        halfgamma = CubicSpline(t, halfgammadot).antiderivative()(t)
        Rgamma = np.stack([np.cos(halfgamma), 0 * halfgamma, 0 * halfgamma, np.sin(halfgamma)], axis=-1)
        R = Q.qmul(R, Rgamma)
    return R


def rotor_angular_velocity(R, t):
    """omega = 2 (dR/dt) R^-1 of a rotor series, dR/dt from cubic splines (quaternion.angular_velocity as called at
    scri/rotations.py:42)."""
    from scipy.interpolate import CubicSpline

    R = np.asarray(R, dtype=float)
    Rdot = CubicSpline(t, R).derivative()(t)
    return (2 * Q.qmul(Rdot, Q.qconj(R)))[:, 1:]


def inner_product(t, abar, b, axis=None, apply_conjugate=False):
    """Spline definite integral over t[0]..t[-1] of abar * b (conj(abar) * b with `apply_conjugate`), elementwise - no sum
    over modes (scri/mode_calculations.py:493-534, quaternion.calculus.spline_definite_integral).

    `axis` is the time axis of the (broadcast) integrand; None takes the first axis whose length is t.size.  The result has
    the integrand's shape without that axis (a 0-d array for 1-D input); it is complex unless both inputs are real.  Device
    tensors stay on the device (a tensor result), host arrays give numpy.  The integrand is never formed: the time axis is
    moved to the front and every remaining element is one column of a weighted streaming sum (csrc/inner.cu)."""
    _lib.require_cuda()
    t = np.asarray(ops.to_host(t), dtype=float).ravel()
    on_device = ops.is_tensor(abar) or ops.is_tensor(b)
    if on_device:
        import torch

        x, y = (v if ops.is_tensor(v) else torch.as_tensor(np.asarray(v)) for v in (abar, b))
        x, y = x.cuda(), y.cuda()
        x, y = torch.broadcast_tensors(x, y)
        is_complex = x.is_complex() or y.is_complex()
    else:
        x, y = np.broadcast_arrays(np.asarray(abar), np.asarray(b))
        is_complex = np.iscomplexobj(x) or np.iscomplexobj(y)
    shape = tuple(x.shape)
    if axis is None:
        axes = [i for i, n in enumerate(shape) if n == t.size]
        if not axes:
            raise ValueError(f"inner_product: no axis of the integrand (shape {shape}) has the length of t ({t.size})")
        axis = axes[0]
    axis = int(axis) % len(shape)
    if shape[axis] != t.size:
        raise ValueError(f"inner_product: axis {axis} of the integrand (shape {shape}) does not have the length of t ({t.size})")
    w = ops.spline_integral_weights_device(t)
    N = t.size
    rest = shape[:axis] + shape[axis + 1:]
    if on_device:
        xm, ym = (v.movedim(axis, 0).reshape(N, -1) for v in (x, y))
    else:
        xm, ym = (np.ascontiguousarray(np.moveaxis(v, axis, 0).reshape(N, -1), dtype=np.complex128) for v in (x, y))
    if xm.shape[1] == 0:
        out = np.zeros(rest, dtype=complex if is_complex else float)
        return torch.from_numpy(out).cuda() if on_device else out
    out = ops.inner_product(xm, ym, w, conjugate=apply_conjugate, per_column=True)
    out = out.reshape(rest)
    return out if is_complex else out.real


def inner_product_matrix(t, a, b, t1=None, t2=None):
    """G [P, Q] complex128 with G[p, q] = the inner product of waveform p of `a` with waveform q of `b` - exactly
    `WaveformModes.inner_product` of that pair: integral from t1 to t2 (default: the first and last time) of
    sum_m conj(a[p, :, m]) b[q, :, m] through the not-a-knot cubic spline of the samples `t`.

    Not in scri: a project extension for comparing batches (e.g. the [B, N', n] output of parallel.transform_batch) without
    bringing them back to the host.  a [P, N, n], b [Q, N, n] (or [N, n] for one waveform): numpy arrays or device tensors;
    a tensor result for tensor input.  One sum per pair on the FP64 tensor cores (P, Q > 1) or the streaming kernel (a single
    row or column of G), csrc/inner.cu."""
    _lib.require_cuda()
    t = np.asarray(ops.to_host(t), dtype=float).ravel()
    for name, v in (("a", a), ("b", b)):
        if tuple(v.shape)[-2] != t.size:
            raise ValueError(f"inner_product_matrix: {name} of shape {tuple(v.shape)} does not have {t.size} time samples on axis -2")
    w = ops.spline_integral_weights_device(t, t1, t2)
    return ops.inner_product_matrix(a, b, w)
