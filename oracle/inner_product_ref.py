"""CPU restatement of scri's time-domain inner products (reference: moble/scri v2024.0.13,
scri/mode_calculations.py:493-534 and scri/waveform_modes.py:574-656).

TEST INFRASTRUCTURE (see oracle/__init__.py) - never imported by scri_b200/.

No golden vector covers these two functions: they are pinned by this literal restatement of the reference flow on the
refshim `quaternion.calculus.spline_definite_integral` (InterpolatedUnivariateSpline(t, f, k=3).integral per real part, as
numpy-quaternion does with scipy present).  Waveforms are the oracle's `Modes` records (oracle/scri_ref.py).
"""
import numpy as np
from scipy.interpolate import CubicSpline


def _refshim_calculus():
    """oracle/refshim/quaternion/calculus.py, loaded by path: importing the `quaternion` stand-in package would also install
    its rotor-aware numpy predicates, which only the golden-vector generation wants."""
    import importlib.util
    import os
    import sys

    name = "oracle._refshim_quaternion_calculus"
    mod = sys.modules.get(name)
    if mod is None:
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "refshim", "quaternion", "calculus.py")
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        sys.modules[name] = mod
    return mod


def inner_product(t, abar, b, axis=None, apply_conjugate=False):
    # mode_calculations.py:493-534: the integrand is elementwise (no sum over modes), integrated over all of t
    if apply_conjugate:
        integrand = np.conj(abar) * b
    else:
        integrand = abar * b
    return _refshim_calculus().spline_definite_integral(integrand, t, axis=axis)


def waveform_inner_product(a, b, t1=None, t2=None, allow_LM_differ=False, allow_times_differ=False, intersection=None):
    """waveform_modes.py:574-656 on `Modes` records.  `intersection` is scri/extrapolation.py:47-125 (needed only when the
    time axes differ): the caller passes an implementation pinned against the reference's own output."""
    if a.spin_weight != b.spin_weight:
        raise ValueError("Spin weights must match in inner_product")
    LM_clip = None
    if (a.ell_min != b.ell_min) or (a.ell_max != b.ell_max):
        if allow_LM_differ:
            LM_clip = slice(max(a.ell_min, b.ell_min), min(a.ell_max, b.ell_max) + 1)
            if LM_clip.start >= LM_clip.stop:
                raise ValueError("Intersection of (ell,m) modes is empty.  Assuming this is not desired.")
        else:
            raise ValueError("ell_min and ell_max must match in inner_product (use allow_LM_differ=True to override)")
    t_clip = None
    if not np.array_equal(a.t, b.t):
        if allow_times_differ:
            t_clip = intersection(a.t, b.t)
        else:
            raise ValueError("Time samples must match in inner_product (use allow_times_differ=True to override)")
    times, A, B = a.t, a.data, b.data
    if LM_clip is not None:
        # WaveformModes.__getitem__ with an ell slice (waveform_modes.py:953-1021): columns of ell_lo .. ell_hi - 1
        lo, hi = LM_clip.start, LM_clip.stop - 1
        A = A[:, lo**2 - a.ell_min**2 : hi * (hi + 2) + 1 - a.ell_min**2]
        B = B[:, lo**2 - b.ell_min**2 : hi * (hi + 2) + 1 - b.ell_min**2]
    if t_clip is not None:
        # WaveformModes.interpolate (waveform_base.py:949-967): a not-a-knot CubicSpline of the data
        times = t_clip
        A, B = CubicSpline(a.t, A)(t_clip), CubicSpline(b.t, B)(t_clip)
    if t1 is None:
        t1 = times[0]
    if t2 is None:
        t2 = times[-1]
    integrand = np.sum(np.conj(A) * B, axis=1)
    return _refshim_calculus().spline_definite_integral(integrand, times, t1=t1, t2=t2)
