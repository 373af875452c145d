"""CPU-side tests of the product's host logic: table builders, kwargs processing, API shell, C-ABI exports."""
import ctypes
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

import scri_b200 as sb
from scri_b200 import _lib, _sf, flux, ops, plan
from scri_b200 import _quaternion as Q
from oracle import quat, scri_ref as R, sf as osf, spinsfast as ospf
from scri_inputs import real_supertranslation, rotor_set, smooth_modes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_lm_layout_bit_exact():
    """(ell,m) indexing must be bit-exact (scri/waveform_modes.py:404-455)."""
    for lmin, lmax in [(0, 4), (2, 8), (1, 16)]:
        LM = _sf.LM_range(lmin, lmax)
        assert np.array_equal(LM, osf.LM_range(lmin, lmax))
        assert LM.shape[0] == _sf.LM_total_size(lmin, lmax)
        for i, (l, m) in enumerate(LM):
            assert _sf.LM_index(l, m, lmin) == i
        for l in range(lmin, lmax + 1):
            assert _sf.D_offset(l, lmin) == osf.linear_matrix_offset(l, lmin)
    w = sb.sample_waveforms.constant_waveform()
    assert w.index(2, -2) == 0 and w.index(8, 8) == 76 and w.n_modes == 77
    with pytest.raises(ValueError):
        w.index(9, 0)


def test_wigner_recurrence_matches_oracle():
    rng = np.random.default_rng(0)
    Rq = quat.normalized(rng.normal(size=(64, 4)))
    Rq[0] = [1, 0, 0, 0]; Rq[1] = [0, 0, 1, 0]; Rq[2] = [0, 1, 0, 0]; Rq[3] = [0, 0, 0, 1]
    Rq[4] = quat.normalized([1, 1e-9, 0, 0]); Rq[5] = quat.normalized([1e-9, 1e-10, 1, 0.3])
    sp = quat.as_spinor_array(Rq)
    for lmin, lmax in [(0, 12), (2, 8)]:
        A = osf.Wigner_D_matrices(sp[:, 0], sp[:, 1], lmin, lmax)
        B = _sf.wigner_D_matrices(sp[:, 0], sp[:, 1], lmin, lmax)
        assert abs(A - B).max() < 2e-14
    for s in (-2, 0, 1, 2):
        assert abs(osf.SWSH_grid(Rq, s, 12) - _sf.SWSH_grid(Rq, s, 12)).max() < 2e-14


@pytest.mark.parametrize("s,lmax,nth,nph", [(-2, 8, 19, 19), (-2, 8, 25, 25), (0, 4, 9, 9), (1, 5, 13, 11), (2, 6, 14, 16)])
def test_analysis_tables_equal_huffenberger_wandelt(s, lmax, nth, nph):
    """phi-DFT + Clenshaw-Curtis theta quadrature == the oracle's literal H&W map2salm, also on white noise."""
    rng = np.random.default_rng(5)
    f = rng.normal(size=(3, nth, nph)) + 1j * rng.normal(size=(3, nth, nph))
    a = ospf.map2salm(f, s, lmax)
    E, Wt = _sf.analysis_tables(s, 0, lmax, nth, nph)
    fm = np.einsum("bjk,km->bjm", f, E)
    b = np.zeros_like(a)
    for l in range(lmax + 1):
        for m in range(-l, l + 1):
            b[:, l * (l + 1) + m] = fm[:, :, m + lmax] @ Wt[l * (l + 1) + m]
    assert abs(a - b).max() < 1e-14


def test_process_transformation_kwargs_matches_oracle():
    kw = dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03])
    a = plan.process_transformation_kwargs(8, **dict(kw))
    b = R.process_transformation_kwargs(8, **dict(kw))
    assert np.array_equal(a[0], b[0]) and a[1:5] == b[1:5]
    assert a[7] == b[7] and a[8] == b[8]
    assert abs(a[9] - b[9]).max() < 1e-15          # rotor grid
    for kw2 in (dict(time_translation=1.5), dict(space_translation=[0.1, -0.2, 0.3]), dict(spacetime_translation=[1.0, 2.0, 3.0, 4.0]), {}):
        a = plan.process_transformation_kwargs(8, **dict(kw2))
        b = R.process_transformation_kwargs(8, **dict(kw2))
        assert np.allclose(a[0], b[0], rtol=0, atol=0) and a[2:5] == b[2:5] and abs(a[9] - b[9]).max() < 1e-15


def test_process_transformation_kwargs_errors():
    """Same exception types as scri/waveform_grid.py:28-125."""
    with pytest.raises(ValueError):
        plan.process_transformation_kwargs(8, supertranslation=np.zeros(7))      # not a perfect square
    bad = np.zeros(9, complex); bad[5] = 1.0
    with pytest.raises(ValueError):
        plan.process_transformation_kwargs(8, supertranslation=bad)               # imaginary supertranslation
    with pytest.raises(TypeError):
        plan.process_transformation_kwargs(8, time_translation=1)                 # int, not float
    with pytest.raises(TypeError):
        plan.process_transformation_kwargs(8, space_translation=[1.0, 2.0])
    with pytest.raises(ValueError):
        plan.process_transformation_kwargs(8, boost_velocity=[1.0, 0.0, 0.0])
    with pytest.raises(ValueError):
        plan.process_transformation_kwargs(8, frame_rotation=[0.0, 0.0, 0.0, 0.0])
    with pytest.raises(ValueError):
        plan.process_transformation_kwargs(8, n_theta=5)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        plan.process_transformation_kwargs(8, supertranslation=real_supertranslation(2), n_theta=17)
        assert any("n_theta" in str(r.message) for r in rec)


def test_pack_synthesis_matrix_is_the_complex_product():
    rng = np.random.default_rng(2)
    G, lmin, lmax = 11, 2, 4
    Y = rng.normal(size=(G, (lmax + 1) ** 2)) + 1j * rng.normal(size=(G, (lmax + 1) ** 2))
    B, Kpad, Ncpad = plan.pack_synthesis_matrix(Y, lmin, lmax)
    n = _sf.LM_total_size(lmin, lmax)
    a = rng.normal(size=(5, n)) + 1j * rng.normal(size=(5, n))
    A = np.zeros((5, Kpad)); A[:, : 2 * n] = a.view(float)
    C = (A @ B)[:, : 2 * G].copy().view(complex)
    assert np.allclose(C, a @ Y[:, lmin * lmin :].T, rtol=1e-13)
    assert Kpad % 16 == 0 and Ncpad % 64 == 0


def test_flux_matrices_match_oracle():
    for lmin, lmax in [(2, 8), (2, 5)]:
        for mine, ref in [
            (flux.p_z(lmin, lmax, s=-2), R.p_z(lmin, lmax, -2)),
            (flux.p_plus(lmin, lmax, s=-2), R.p_plusminus(lmin, lmax, +1, -2)),
            (flux.p_minus(lmin, lmax, s=-2), R.p_plusminus(lmin, lmax, -1, -2)),
            (flux.j_z(lmin, lmax), R.j_z(lmin, lmax)),
            (flux.j_plus(lmin, lmax), R.j_plusminus(lmin, lmax, +1)),
            (flux.j_minus(lmin, lmax), R.j_plusminus(lmin, lmax, -1)),
        ]:
            assert np.array_equal(mine[0], ref[0]) and np.array_equal(mine[1], ref[1])
            assert np.allclose(mine[2], ref[2], rtol=1e-14, atol=1e-15)


def test_quaternion_helpers_match_oracle():
    rng = np.random.default_rng(3)
    p, q = rng.normal(size=(2, 20, 4))
    assert np.allclose(Q.qmul(p, q), quat.mul(p, q))
    assert np.allclose(Q.as_spinor_array(p), quat.as_spinor_array(p))
    u = Q.qnormalized(p)
    assert np.allclose(Q.rotate_z(u), quat.rotate_vector(u, np.array([0.0, 0.0, 1.0])))
    th, ph = Q.as_spherical_coords(u)
    assert np.allclose(np.stack([th, ph], -1), quat.as_spherical_coords(u))
    assert np.allclose(Q.qmul(Q.qsqrt(u), Q.qsqrt(u)), u)


def test_sample_waveforms_host_side():
    w = sb.sample_waveforms.fake_precessing_waveform(t_1=500.0, inertial=False)
    assert w.frameType == sb.Corotating and w.dataType == sb.h and w.n_modes == 77
    assert not np.isnan(w.data).any() and w.frame.shape == (w.n_times, 4)
    assert np.allclose(np.sum(w.frame**2, axis=1), 1.0)
    # conjugate-pair structure of the PN amplitudes: h_{l,-m} = (-1)^l conj(h_{l,m}) up to the modulation
    a = sb.sample_waveforms.pn_leading_order_amplitude(3, 2, 0.1, 2.0)
    b = sb.sample_waveforms.pn_leading_order_amplitude(3, -2, 0.1, 2.0)
    assert np.isclose(b, (-1) ** 3 * np.conj(a))
    t, batch = sb.sample_waveforms.smooth_random_waveform(n_times=64, batch=3)
    assert batch.shape == (3, 64, 77)


def test_waveform_shell_history_copy_and_validity():
    w = sb.sample_waveforms.constant_waveform()
    c = w.copy()
    assert c is not w and np.array_equal(c.data, w.data) and c.ell_min == 2 and c.ell_max == 8
    assert c.spin_weight == -2 and c.conformal_weight == -1 and c.data_type_string == "h" and c.frame_type_string == "Inertial"
    assert any("copy()" in line for line in c.history)
    with pytest.raises(ValueError):
        sb.WaveformModes(t=np.array([0.0, 1.0, 1.0]), data=np.zeros((3, 77), complex), ell_min=2, ell_max=8)
    with pytest.raises(ValueError):
        sb.WaveformModes(t=np.arange(3.0), data=np.zeros((3, 70), complex), ell_min=2, ell_max=8)
    with pytest.raises(TypeError):
        sb.WaveformGrid.from_modes("not a waveform")
    corot = sb.WaveformModes(t=np.arange(5.0), data=np.zeros((5, 77), complex), ell_min=2, ell_max=8, frameType=sb.Corotating, dataType=sb.h)
    with pytest.raises(ValueError):
        corot.transform(time_translation=1.0)     # must be inertial (scri/waveform_grid.py:422-426)


def test_no_cpu_fallback():
    """Without a CUDA device the operators must fail loudly rather than compute on the CPU.  On a machine with a device
    this test runs again in a child process that is shown none."""
    import torch

    if torch.cuda.is_available():
        child = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", f"{__file__}::test_no_cpu_fallback"],
                               cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
        assert child.returncode == 0 and "1 passed" in child.stdout, child.stdout + child.stderr
        return
    w = sb.sample_waveforms.constant_waveform()
    with pytest.raises(_lib.Scrib200Error):
        w.transform(time_translation=1.0)
    with pytest.raises(_lib.Scrib200Error):
        w.rotate_decomposition_basis(np.array([1.0, 0.0, 0.0, 0.0]))
    with pytest.raises(_lib.Scrib200Error):
        w.LLMatrix()


def test_product_never_imports_the_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "scri_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"


def test_c_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "scrib200.h")).read()
    declared = set(re.findall(r"\b(scrib200_[a-z0-9_]+)\s*\(", header))
    assert declared, "no declarations parsed"
    assert os.path.exists(_lib.LIB_PATH), "libscrib200.so not built (run __graft_entry__.build())"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/scrib200.h but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib.scrib200_version.restype = ctypes.c_int
    assert lib.scrib200_version() >= 100


def test_ladder_table():
    tab = ops.ladder_table(2, 4)
    LM = _sf.LM_range(2, 4)
    for row, (l, m) in zip(tab, LM):
        assert row[4] == m
        assert np.isclose(row[0], np.sqrt((l - m) * (l + m + 1)) if m + 1 <= l else 0.0)
        assert np.isclose(row[1], np.sqrt((l + m) * (l - m + 1)) if m - 1 >= -l else 0.0)


@pytest.mark.parametrize("case", [(2, 3, -2, 4, None, None), (0, 4, 1, 2, None, 6), (2, 5, -2, 5, 6, 4), (-1, 3, 0, 3, 3, 3)])
def test_product_tables_through_a_numpy_emulation_of_the_kernel(case):
    """Host tables of the fused separable product (scri_b200/_product.py: mode permutation, DMMA fragment order of the
    Wigner-d and quadrature tables, alias range of the m-convolution) drive a numpy emulation of csrc/product.cu's
    three stages; the result is ModesTimeSeries.grid_multiply's (scri/modes_time_series.py:142-202), aliased working
    grids (working_ell_max < ell1 + ell2) included."""
    from oracle import abd_ref
    from product_emulator import emulate
    from scri_b200 import _product

    s1, L1, s2, L2, Lw, Lo = case
    rng = np.random.default_rng(0)

    def rnd(L, s):
        a = rng.normal(size=(6, (L + 1) ** 2)) + 1j * rng.normal(size=(6, (L + 1) ** 2))
        a[:, : s * s] = 0
        return a

    a, b = rnd(L1, s1), rnd(L2, s2)
    ref = abd_ref.grid_multiply(a, s1, b, s2, working_ell_max=Lw, output_ell_max=Lo)
    n = 2 * (L1 + L2 if Lw is None else Lw) + 1
    for shape in (None, 1, 2):   # default, 8-warp and cluster (CTA pair) table sets
        tb = _product.product_tables(s1, 0, L1, s2, 0, L2, n, n, L1 if Lo is None else Lo, shape)
        assert tb.fits
        assert np.abs(emulate(tb, a, b) - ref).max() < 1e-14 * np.abs(ref).max()


def test_product_tables_config4_fit_one_cta():
    from scri_b200 import _product

    tb = _product.product_tables(2, 0, 32, -2, 0, 32, 129, 129, 32)
    assert tb.fits and tb.smem_bytes <= 227 * 1024 and (tb.gm, tb.nwarps) == (5, 16)
    assert _product.product_tables(2, 0, 32, -2, 0, 32, 129, 129, 32, shape=1).nwarps == 8
    assert not _product.product_tables(2, 0, 64, -2, 0, 64, 257, 257, 64).fits   # the dense kernels take over


def test_native_rotor_integrator_against_closed_form_and_scipy():
    """scrib200_integrate_angular_velocity (host code of the library; quaternion.integrate_angular_velocity at
    scri/mode_calculations.py:467): a constant angular velocity has the closed form exp(omega t / 2); a precessing one is
    compared with scipy's DOP853 at a tighter tolerance.  The reference's own bar for the corotating frame is 1e-10
    (tests/test_rotations.py); the native integrator clips its steps to the samples and lands well inside it."""
    from scipy.integrate import solve_ivp
    from scipy.interpolate import CubicSpline

    from scri_b200 import mode_calculations as mc

    t = np.arange(-20.0, 400.0, 0.1)
    om_c = np.tile(np.array([0.1, -0.2, 0.3]), (t.size, 1))
    th = np.linalg.norm(om_c[0]) * (t - t[0]) / 2
    n = om_c[0] / np.linalg.norm(om_c[0])
    exact = np.stack([np.cos(th), n[0] * np.sin(th), n[1] * np.sin(th), n[2] * np.sin(th)], axis=1)
    assert np.abs(mc.integrate_angular_velocity(t, om_c) - exact).max() < 1e-12
    w0 = 0.05 + 0.4 * ((t - t[0]) / (t[-1] - t[0])) ** 3
    omega = np.stack([0.02 * np.cos(0.01 * t) * w0, 0.02 * np.sin(0.01 * t) * w0, w0], axis=1)
    R0 = Q.qnormalized(np.array([1.0, 2.0, 3.0, 4.0]))
    Rn = mc.integrate_angular_velocity(t, omega, R0=R0, tolerance=1e-12)
    assert np.array_equal(Rn[0], R0) and np.abs(np.linalg.norm(Rn, axis=1) - 1).max() < 1e-12
    om = CubicSpline(t, omega)

    def rhs(tt, y):
        w = om(tt)
        return 0.5 * Q.qmul(np.array([0.0, w[0], w[1], w[2]]), y)

    sol = solve_ivp(rhs, (t[0], t[-1]), R0, method="DOP853", t_eval=t[::50], atol=1e-13, rtol=1e-13)
    assert np.abs(sol.y.T - Rn[::50]).max() < 5e-12
    with pytest.raises((ValueError, _lib.Scrib200Error)):
        mc.integrate_angular_velocity(np.array([0.0, 1.0, 1.0, 2.0, 3.0]), np.zeros((5, 3)))      # times must increase


def test_squad_reproduces_knots_and_geodesics():
    """quaternion.squad as used by WaveformBase.interpolate (scri/waveform_base.py:962): the samples are reproduced exactly,
    a uniformly rotating series stays on its geodesic between unevenly spaced samples, and the interpolant of a smooth
    rotation converges."""
    rng = np.random.default_rng(0)
    t = np.sort(rng.uniform(0, 10, 40))
    t[0], t[-1] = 0.0, 10.0
    axis = np.array([0.3, -0.5, 0.8]) / np.linalg.norm([0.3, -0.5, 0.8])
    R0 = Q.qnormalized(np.array([1.0, 2.0, 3.0, 4.0]))

    def geodesic(tt):
        return Q.qmul(Q.qexp_vec(0.35 * tt[:, None] * axis[None, :]), R0[None, :])

    R = geodesic(t)
    assert np.array_equal(Q.squad(R, t, t), R)
    tt = np.linspace(0, 10, 333)
    assert np.abs(Q.squad(R, t, tt) - geodesic(tt)).max() < 1e-13

    def wobble(x):
        ax = np.stack([np.sin(0.2 * x), np.cos(0.2 * x), 0.5 + 0 * x], 1)
        return Q.qexp_vec(0.5 * (0.7 * x + 0.3 * np.sin(x))[:, None] * ax / np.linalg.norm(ax, axis=1)[:, None])

    errs = [np.abs(Q.squad(wobble(np.linspace(0, 10, n)), np.linspace(0, 10, n), tt) - wobble(tt)).max() for n in (50, 100, 200)]
    assert errs[0] > 3 * errs[1] > 9 * errs[2]
    assert Q.squad(np.empty((0, 4)), np.empty(0), tt).shape == (0, 4)


def test_intersection_matches_reference_output():
    """scri/extrapolation.py:47-125 as run by the reference (tests/golden/reference_expectation.npz) vs the host restatement
    scri_b200.flux.intersection used by matrix_expectation_value(allow_times_differ=True): bit for bit."""
    import os

    from scri_b200.flux import intersection

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_expectation.npz"))
    assert np.array_equal(intersection(g["i_t1"], g["i_t2"]), g["i_out"])
    assert np.array_equal(intersection(g["i_t1"], g["i_t2"], min_step=0.9, min_time=5.0, max_time=70.0), g["i_out_kw"])
    with pytest.raises(ValueError):
        intersection(np.array([]), g["i_t2"])
    with pytest.raises(ValueError):
        intersection(g["i_t1"], g["i_t2"] + 1000.0)


def _unpack_fragments(table, offsets, ell):
    """(Delta^T, Delta) of one l rebuilt from the m8n8k4 A-fragment table: lane holds A[8 mm + lane / 4][4 kk + lane % 4]."""
    n = 2 * ell + 1
    Mt, Kt = (n + 7) // 8, (n + 3) // 4
    out = []
    for part in range(2):
        tiles = table[offsets[ell] + part * Mt * Kt * 32 : offsets[ell] + (part + 1) * Mt * Kt * 32].reshape(Kt, Mt, 8, 4)
        A = tiles.transpose(1, 2, 0, 3).reshape(8 * Mt, 4 * Kt)
        assert not A[n:].any() and not A[:, n:].any()            # padding is exactly zero
        out.append(A[:n, :n])
    return out


@pytest.mark.parametrize("ell_min,ell_max", [(2, 8), (0, 16), (3, 11)])
def test_rotation_tables_through_a_numpy_emulation_of_the_dmma_kernel(ell_min, ell_max):
    """scrib200_rotate_modes_dmma in numpy, from the product's own operand table (ops.delta_fragment_tables): unpack the
    fragments, check Delta^l = d^l(pi/2) is orthogonal with the reflection symmetries the factorisation rests on, then run the
    kernel's five steps - phases, Delta^T, phases of beta, Delta, phases - against the oracle's rotation (poles, an exact
    identity and a 1e-9 neighbourhood of a pole included)."""
    table, offsets = ops.delta_fragment_tables(ell_max)
    rng = np.random.default_rng(ell_max)
    n_t = 24
    t, data = smooth_modes(n_times=n_t, ell_min=ell_min, ell_max=ell_max, seed=7)
    Rs = quat.normalized(rng.normal(size=(n_t, 4)))
    Rs[0] = [1.0, 0.0, 0.0, 0.0]
    Rs[1] = [0.0, 0.0, 1.0, 0.0]
    Rs[2] = [0.0, 1.0, 0.0, 0.0]
    Rs[3] = np.array([1e-9, 0.0, 1.0, 0.0]) / np.sqrt(1.0 + 1e-18)
    want = R.rotate_decomposition_basis(R.Modes(t=t, data=data.copy(), ell_min=ell_min, ell_max=ell_max), Rs).data
    sp = Q.as_spinor_array(Rs)
    Ra, Rb = sp[:, 0], sp[:, 1]
    ra2, rb2 = np.abs(Ra) ** 2, np.abs(Rb) ** 2
    n2 = ra2 + rb2
    ea = np.where(ra2 > 0, Ra / np.where(ra2 > 0, np.abs(Ra), 1.0), 1.0)
    eb = np.where(rb2 > 0, Rb / np.where(rb2 > 0, np.abs(Rb), 1.0), 1.0)
    ra, rb = np.sqrt(ra2 / n2), np.sqrt(rb2 / n2)
    q1, ebeta, q3 = -1j * ea * np.conj(eb), (ra * ra - rb * rb) - 2j * ra * rb, 1j * ea * eb
    got = np.empty_like(data)
    for ell in range(ell_min, ell_max + 1):
        dT, d = _unpack_fragments(table, offsets, ell)
        assert np.array_equal(dT, d.T)
        n = 2 * ell + 1
        m = np.arange(-ell, ell + 1)
        assert np.abs(d @ d.T - np.eye(n)).max() < 4e-15
        assert np.array_equal(d[::-1, :], d * (-1.0) ** (ell + m)[None, :])       # Delta[-m', mu] = (-1)^(l + mu) Delta[m', mu]
        assert np.array_equal(d[:, ::-1], d * (-1.0) ** (ell + m)[:, None])       # Delta[m', -mu] = (-1)^(l + m') Delta[m', mu]
        col = ell * ell - ell_min * ell_min
        x = data[:, col : col + n] * q1[:, None] ** m[None, :]
        y = x @ dT.T                                                               # y[mu] = sum_m' Delta[m', mu] x[m']
        z = y * ebeta[:, None] ** m[None, :]
        o = z @ d.T                                                                # o[m] = sum_mu Delta[m, mu] z[mu]
        got[:, col : col + n] = o * q3[:, None] ** m[None, :]
    assert np.abs(got - want).max() / np.abs(want).max() < 2e-14


@pytest.mark.parametrize("same", [True, False])
def test_expectation_tables_through_a_numpy_emulation_of_the_time_lane_kernel(same):
    """ops._time_tables (entry table + column blocks of scrib200_sparse_expectation_time) for the momentum operators at
    ell <= 16: every column with entries lies in exactly one block, every row an entry names (padding slots included) lies in
    its block's window, the tiles fit the budget the way the C side adds them up - and walking the table block by block the
    way the kernel does gives the dense contraction."""
    lmin, lmax = 2, 16
    n = lmax * (lmax + 2) - lmin * lmin + 1
    mats = [flux.p_plus(lmin, lmax, s=-2), flux.p_minus(lmin, lmax, s=-2), flux.p_z(lmin, lmax, s=-2)]
    tab, blocks, width, real = ops._time_tables(mats, n, same)
    blocks = blocks.reshape(-1, 4)
    assert real and width == 3 and tab.shape == (n, 3, 3) and tab.dtype.itemsize == 16
    covered = np.zeros(n, dtype=int)
    for c0, c1, rlo, rhi in blocks:
        covered[c0:c1] += 1
        r = tab["r"][c0:c1]
        assert r.min() >= rlo and r.max() < rhi
        if same:
            assert rlo <= c0 and c1 <= rhi
    assert (covered == 1).all() and len(blocks) >= 2
    max_rows, max_cols = (blocks[:, 3] - blocks[:, 2]).max(), (blocks[:, 1] - blocks[:, 0]).max()
    assert (max_rows + (0 if same else max_cols)) * 528 + max_cols * 9 * 16 <= ops.XT_BUDGET_BYTES
    rng = np.random.default_rng(3)
    a = rng.normal(size=(5, n)) + 1j * rng.normal(size=(5, n))
    b = a if same else rng.normal(size=(5, n)) + 1j * rng.normal(size=(5, n))
    got = np.zeros((5, 3), dtype=complex)
    for c0, c1, rlo, rhi in blocks:
        for c in range(c0, c1):
            for k in range(3):
                q = sum(tab["v"][c, k, w] * np.conj(a[:, tab["r"][c, k, w]]) for w in range(width))
                got[:, k] += q * b[:, c]
    want = np.zeros((5, 3), dtype=complex)
    for k, (rows, cols, vals) in enumerate(mats):
        M = np.zeros((n, n), dtype=complex)
        M[np.asarray(rows), np.asarray(cols)] = vals
        want[:, k] = np.einsum("tr,rc,tc->t", a.conj(), M, b)
    assert np.abs(got - want).max() / np.abs(want).max() < 1e-14

