"""Parity tests proper: the CUDA path (through the Python API -> ctypes -> C ABI) against the CPU oracle, the
committed golden fixtures, and size-independent properties at BASELINE.json's full sizes.  Need a B200."""
import os

import numpy as np
import pytest

import scri_b200 as sb
from scri_b200 import _lib, ops, plan as P
from oracle import quat, scri_ref as R
from scri_inputs import real_supertranslation, rotor_set, smooth_modes

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")

# Floating-point tolerance from BASELINE.json north_star: 1e-12 relative (FP64); measured headroom ~1e-14.
RTOL = 1e-12


def rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def modes(t, data, ell_min=2, ell_max=8, dataType=sb.h, frameType=sb.Inertial, **kw):
    return sb.WaveformModes(t=t, data=data.copy(), ell_min=ell_min, ell_max=ell_max, frameType=frameType, dataType=dataType,
                            r_is_scaled_out=True, m_is_scaled_out=True, **kw)


BMS = dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03])


def test_native_library_is_loaded():
    lib = _lib.load()
    assert lib.scrib200_version() >= 100
    before = _lib.launch_count()
    ops.norm(np.ones((4, 5), complex))
    assert _lib.launch_count() == before + 1


# ------------------------------------------------------------------ rotation (K4)
def test_rotation_series_and_constant_vs_oracle():
    t, data = smooth_modes(n_times=300)
    Rs = quat.normalized(np.random.default_rng(1).normal(size=(300, 4)))
    w = modes(t, data)
    w.rotate_decomposition_basis(Rs)
    Wo = R.rotate_decomposition_basis(R.Modes(t=t, data=data.copy()), Rs)
    assert rel(w.data, Wo.data) < 1e-13
    assert np.allclose(w.frame, Rs)
    w = modes(t, data)
    w.rotate_decomposition_basis(Rs[0])
    Wo = R.rotate_decomposition_basis(R.Modes(t=t, data=data.copy()), Rs[0])
    assert rel(w.data, Wo.data) < 1e-13 and w.frame.shape == (1, 4)


def test_rotation_identity_is_bit_exact_and_inverse_round_trip():
    """reference tests/test_rotations.py:14-129"""
    t, data = smooth_modes(n_times=100)
    w = modes(t, data)
    w.rotate_decomposition_basis(np.array([1.0, 0.0, 0.0, 0.0]))
    assert np.array_equal(w.data, data)
    for Rq in rotor_set(4):
        w = modes(t, data)
        w.rotate_decomposition_basis(Rq)
        assert np.allclose(w.norm(), np.sum(abs(data) ** 2, axis=1), rtol=1e-13)
        w.rotate_decomposition_basis(quat.conj(Rq))
        assert np.allclose(w.data, data, rtol=0, atol=8**4 * 4e-14)
        assert np.allclose(abs(w.frame[0, 0]), 1.0)   # frame * R * ~R = +-1


def test_rotation_poles_and_large_ell():
    t, data = smooth_modes(n_times=12, ell_min=0, ell_max=16, seed=9)
    Rs = np.array([[0, 0, 1.0, 0], [0, 1.0, 0, 0], [0, 0, 0, 1.0], [1e-9, 0, 1.0, 0], [1.0, 1e-9, 0, 0], [0.6, 0, 0, 0.8]] * 2)
    Rs = Rs / np.linalg.norm(Rs, axis=1)[:, None]
    d = data.copy()
    ops.rotate_modes(d, Rs, 0, 16)
    Wo = R.rotate_decomposition_basis(R.Modes(t=t, data=data.copy(), ell_min=0, ell_max=16), Rs)
    assert rel(d, Wo.data) < 1e-12


@pytest.mark.parametrize("recurrence", [False, True])
@pytest.mark.parametrize("ell_min,ell_max", [(2, 8), (2, 16), (0, 16), (0, 8), (3, 11), (10, 14), (2, 5), (13, 16), (9, 12), (2, 12), (1, 1), (0, 0), (2, 20)])
def test_rotation_every_block_instantiation(ell_min, ell_max, recurrence, monkeypatch):
    """rotate.cu has two rotation kernels for ell_max <= 16 - the DMMA kernel (tiles sized for ell_max <= 11 or <= 16, 1..5
    m-tiles per l) and the recurrence kernel (one launch per block of l: 0..8, 9..12, 13..16, in an instantiation without
    per-rung tests when the block is covered completely and a general one otherwise; SCRIB200_ROTATE_RECURRENCE) - and the
    first-generation kernel above: every combination against the oracle, on a series that does not fill its last tile
    and contains an exact identity and an exact pole."""
    if recurrence:
        monkeypatch.setenv("SCRIB200_ROTATE_RECURRENCE", "1")
    n = 77
    t, data = smooth_modes(n_times=n, ell_min=ell_min, ell_max=ell_max, seed=31 + ell_min + 17 * ell_max)
    Rs = quat.normalized(np.random.default_rng(ell_max).normal(size=(n, 4)))
    Rs[5] = [1.0, 0.0, 0.0, 0.0]
    Rs[40] = [0.0, 1.0, 0.0, 0.0]
    d = data.copy()
    ops.rotate_modes(d, Rs, ell_min, ell_max)
    Wo = R.rotate_decomposition_basis(R.Modes(t=t, data=data.copy(), ell_min=ell_min, ell_max=ell_max), Rs)
    assert rel(d, Wo.data) < 1e-12
    assert np.array_equal(d[5], data[5])


def test_rotation_full_size_round_trip():
    """1e5 steps (config sizes): R(t) then ~R(t) restores the modes; norm invariant."""
    N = 100_000
    t, data = smooth_modes(n_times=N, t0=0.0, t1=1e4, seed=2)
    rng = np.random.default_rng(3)
    Rs = quat.normalized(rng.normal(size=(N, 4)))
    d = data.copy()
    ops.rotate_modes(d, Rs, 2, 8)
    assert np.allclose(np.sum(abs(d) ** 2, 1), np.sum(abs(data) ** 2, 1), rtol=1e-12)
    ops.rotate_modes(d, quat.conj(Rs), 2, 8)
    assert rel(d, data) < 1e-13


# ------------------------------------------------------------------ transform stages (K1, K2, K3)
def test_transform_stage_by_stage_vs_oracle():
    t, data = smooth_modes(n_times=801, t0=0.0, t1=80.0)
    g_o, inter = R.from_modes(R.Modes(t=t, data=data.copy()), return_intermediates=True, **BMS)
    pl = P.TransformPlan(2, 8, sb.h, **BMS)
    assert rel(pl.kconformal, inter["kconformal"].ravel()) < 1e-15
    assert rel(pl.alpha, inter["alpha"].ravel()) < 1e-14
    td, ad = ops.to_device(t), ops.to_device(data)
    F = pl.synthesize(ad)
    assert rel(F.cpu().numpy(), inter["synthesized"].reshape(len(t), -1)) < 1e-13
    up = pl.output_times(td)
    assert np.array_equal(up.cpu().numpy(), g_o.t)           # output time grid: bit-exact
    grid = pl.remap(td, F, up)
    assert rel(grid.cpu().numpy(), g_o.data) < 1e-13
    for body, halo in ((48, 32), (96, 64), (320, 32), (16, 128), (128, 128)):   # tiling logic: every tiling gives the same spline
        pl.spline_body, pl.spline_halo = body, halo
        assert rel(pl.remap(td, F, up).cpu().numpy(), g_o.data) < 1e-13
    pl.spline_body = pl.spline_halo = 0
    m_o = R.to_modes(g_o, 8)
    assert rel(pl.analyze(grid).cpu().numpy(), m_o.data) < 1e-13
    # analysis alone on the oracle's grid, all modes from ell=0 as spinsfast returns them
    from oracle import spinsfast as ospf
    full = ospf.map2salm(g_o.data.reshape(-1, g_o.n_theta, g_o.n_phi)[:40], -2, 8)
    mine = ops.map2salm(g_o.data.reshape(-1, g_o.n_theta, g_o.n_phi)[:40], -2, 8)
    assert rel(mine, full) < 1e-13


@pytest.mark.parametrize("dataType", [sb.h, sb.sigma, sb.psi4, sb.news])
@pytest.mark.parametrize("uniform", [True, False])
def test_transform_vs_oracle(dataType, uniform):
    s = sb.SpinWeights[dataType]
    t, data = smooth_modes(n_times=500, ell_min=abs(s), uniform=uniform, seed=5)
    w = modes(t, data, ell_min=abs(s), dataType=dataType)
    out = w.transform(**BMS)
    ref = R.transform(R.Modes(t=t, data=data.copy(), ell_min=abs(s), dataType=dataType), **BMS)
    assert np.array_equal(out.t, ref.t)
    assert out.ell_min == abs(s) and out.ell_max == 8 and out.dataType == dataType
    assert rel(out.data, ref.data) < RTOL


@pytest.mark.parametrize("dataType", [sb.psi0, sb.psi1, sb.psi2, sb.psi3])
def test_transform_weyl_scalars_vs_oracle(dataType):
    """psi0..psi3 mix with every higher Weyl scalar under supertranslations and boosts (scri/waveform_grid.py:504-550)."""
    t = np.linspace(-10.0, 100.0, 400)
    ws, wo = {}, {}
    for DT in range(dataType, sb.psi4 + 1):
        s = sb.SpinWeights[DT]
        _, d = smooth_modes(n_times=400, ell_min=abs(s), seed=40 + DT)
        ws[DT] = modes(t, d, ell_min=abs(s), dataType=DT)
        wo[DT] = R.Modes(t=t, data=d.copy(), ell_min=abs(s), dataType=DT)
    extra = {"psi{}_modes".format(sb.DataNames[DT][-1]): ws[DT] for DT in range(dataType + 1, sb.psi4 + 1)}
    extra_o = {"psi{}_modes".format(sb.DataNames[DT][-1]): wo[DT] for DT in range(dataType + 1, sb.psi4 + 1)}
    out = ws[dataType].transform(**BMS, **extra)
    ref = R.transform(wo[dataType], **BMS, **extra_o)
    assert np.array_equal(out.t, ref.t)
    assert out.dataType == dataType and out.ell_min == abs(sb.SpinWeights[dataType])
    assert rel(out.data, ref.data) < RTOL


def test_transform_golden_fixture():
    g = np.load(os.path.join(GOLD, "transform_small.npz"))
    w = modes(g["t"], g["data"])
    out = w.transform(supertranslation=g["supertranslation"], frame_rotation=g["frame_rotation"], boost_velocity=g["boost_velocity"])
    assert np.array_equal(out.t, g["out_t"])
    assert rel(out.data, g["out_data"]) < RTOL


def test_time_translation():
    """reference tests/test_waveform_grid.py:17-27"""
    import math

    dt = 1.469
    w1 = sb.sample_waveforms.constant_waveform()
    w2 = w1.transform(time_translation=dt)
    w3 = w1.transform(supertranslation=[math.sqrt(4 * math.pi) * dt])
    assert np.allclose(w1.t, w2.t + dt, rtol=0.0, atol=2e-15)
    assert np.allclose(w1.data, w2.data, rtol=0.0, atol=4e-14)
    assert np.array_equal(w2.t, w3.t) and np.array_equal(w2.data, w3.data)


def test_BMS_rotation():
    """reference tests/test_waveform_grid.py:30-38"""
    w1 = sb.sample_waveforms.constant_waveform()
    for Rq in rotor_set():
        w2 = w1.copy()
        w2.rotate_decomposition_basis(Rq)
        w3 = w1.transform(frame_rotation=Rq)
        assert np.allclose(w2.data, w3.data, rtol=1e-15, atol=4e-13)


def test_supertranslation_and_boost_inverses():
    """reference tests/test_waveform_grid.py:161-214: T(a) then T(-a), B(v) then B(-v) restore the waveform
    (linear-in-time random modes for the supertranslation, a rotating (2,2) mode for the boost, as there)."""
    rng = np.random.default_rng(4)
    c = rng.normal(size=77) + 1j * rng.normal(size=77)
    t = np.linspace(-10.0, 30.0, 401)
    w1 = modes(t, c[None, :] * t[:, None], dataType=sb.psi4)
    st = real_supertranslation(4, seed=8, scale=0.2)
    w2 = w1.transform(supertranslation=st).transform(supertranslation=-st)
    expect = ops.spline_calculus(w1.t, w1.data, "evaluate", tprime=w2.t)
    assert np.allclose(w2.data, expect, rtol=5e-10, atol=5e-12)
    t = np.arange(-10.0, 10.0, 1.0 / 200.0)
    data = np.zeros((t.size, 77), complex)
    data[:, 4] = np.exp(-2j * 0.3 * t)          # (2,2) mode rotating at omega = 0.3
    w1 = modes(t, data).transform(space_translation=[0.1, 0.0, 0.0])
    w1.m_is_scaled_out = False
    for v in ([0.0, 0.0, 1e-2], [0.0, 1e-2, 0.0], [1e-2, 0.0, 0.0]):
        w2 = w1.transform(boost_velocity=v, n_theta=2 * 9 + 1, n_phi=2 * 9 + 1, ell_max=8)
        w2 = w2.transform(boost_velocity=[-x for x in v], ell_max=8)
        expect = ops.spline_calculus(w1.t, w1.data, "evaluate", tprime=w2.t)
        assert np.allclose(w2.data, expect, rtol=0, atol=1e-12)


def test_to_grid_from_grid_round_trip():
    """config 1 (reduced length here; full length in test_full_size_*): to_grid() / from_grid(ell_max)."""
    w = sb.sample_waveforms.fake_precessing_waveform(t_1=300.0)
    g = w.to_grid()
    assert g.n_theta == 19 and g.n_phi == 19 and g.data.shape == (w.n_times, 361)
    back = sb.WaveformModes.from_grid(g, 8)
    assert np.array_equal(back.t, w.t)
    assert np.allclose(back.data, w.data, rtol=0, atol=1e-13)
    go = R.from_modes(R.Modes(t=w.t, data=w.data.copy()))
    assert rel(g.data, go.data) < 1e-13


def test_edge_cases():
    t, data = smooth_modes(n_times=4)                      # minimum length for a cubic spline
    out = modes(t, data).transform(time_translation=0.0)
    ref = R.transform(R.Modes(t=t, data=data.copy()), time_translation=0.0)
    assert np.array_equal(out.t, ref.t) and rel(out.data, ref.data) < 1e-12
    with pytest.raises(_lib.Scrib200Error):
        modes(t[:3], data[:3]).transform(time_translation=0.0)
    t, data = smooth_modes(n_times=64)
    big = real_supertranslation(2, scale=30.0)             # supertranslation larger than the time span: nothing survives
    out = modes(t, data, dataType=sb.psi4).transform(supertranslation=big)
    ref = R.transform(R.Modes(t=t, data=data.copy(), dataType=R.psi4), supertranslation=big) if False else None
    assert out.n_times <= t.size
    with pytest.raises(ValueError, match="requires information from Psi2"):     # waveform_grid.py:529
        modes(t, np.zeros((64, 80), complex), ell_min=1, ell_max=8, dataType=sb.psi1).transform(boost_velocity=[0.1, 0, 0])


# ------------------------------------------------------------------ full-size properties (config 2)
def test_full_size_transform_inverse_round_trip():
    """1e5 time steps, l<=8: transform with (supertranslation+boost+rotation) then with the inverse rotation/
    time structure checked through invariants the domain offers: (i) the spline does not depend on the tiling,
    (ii) a pure rotation through the BMS path equals the Wigner-D path, (iii) oracle parity on a window."""
    N = 100_000
    t = np.linspace(0.0, 1e4, N)
    _, data = smooth_modes(n_times=N, t0=0.0, t1=1e4, seed=6)
    pl = P.TransformPlan(2, 8, sb.h, **BMS)
    td, ad = ops.to_device(t), ops.to_device(data)
    up, out = pl.run(td, ad)
    pl2 = P.TransformPlan(2, 8, sb.h, **BMS)
    pl2.spline_body, pl2.spline_halo = 160, 64
    up2, out2 = pl2.run(td, ad)
    assert np.array_equal(up.cpu().numpy(), up2.cpu().numpy())
    assert rel(out.cpu().numpy(), out2.cpu().numpy()) < 1e-14
    # oracle on the first 3000 samples (a boosted window must start near t=0 or u'min > u'max); the spline
    # coupling decays as 0.268^k, so outputs 500 samples away from the window's artificial right end are exact
    lo, hi = 0, 3_000
    ref = R.transform(R.Modes(t=t[lo:hi], data=data[lo:hi].copy()), **BMS)
    assert ref.t.shape[0] > 1500
    upn = up.cpu().numpy()
    sel = np.searchsorted(upn, ref.t[:-500])
    assert np.array_equal(upn[sel], ref.t[:-500])
    assert rel(out.cpu().numpy()[sel], ref.data[:-500]) < RTOL
    # rotation only
    Rq = quat.normalized(np.array([1.0, 2.0, 3.0, 4.0]))
    plr = P.TransformPlan(2, 8, sb.h, frame_rotation=Rq)
    _, outr = plr.run(td, ad)
    d = ad.clone()
    ops.rotate_modes(d, Rq, 2, 8)
    assert rel(outr.cpu().numpy(), d.cpu().numpy()) < 1e-13


# ------------------------------------------------------------------ spline calculus, mode calculations, fluxes
def test_modes_golden_fixture():
    g = np.load(os.path.join(GOLD, "modes_small.npz"))
    t, data = g["t"], g["data"]
    w = modes(t, data, ell_max=6)
    d = data.copy()
    ops.rotate_modes(d, g["rotors"], 2, 6)
    assert rel(d, g["rotated"]) < 1e-13
    assert rel(w.data_dot, g["data_dot"]) < 1e-12
    assert rel(w.LLMatrix(), g["LL"]) < 1e-13
    assert rel(w.LdtVector(), g["Ldt"]) < 1e-12
    assert rel(w.LVector(), g["Lvec"]) < 1e-13
    assert np.abs(w.LLDominantEigenvector() - g["dpa"]).max() < 1e-11
    assert rel(w.angular_velocity(), g["omega"]) < 1e-11
    assert rel(w.energy_flux(), g["energy_flux"]) < 1e-12
    assert rel(w.momentum_flux(), g["momentum_flux"]) < 1e-12
    assert rel(w.angular_momentum_flux(), g["angular_momentum_flux"]) < 1e-12


def test_spline_calculus_vs_scipy():
    from scipy.interpolate import CubicSpline

    for uniform in (True, False):
        t, data = smooth_modes(n_times=700, uniform=uniform, seed=21)
        assert rel(ops.spline_calculus(t, data, "derivative", 1), CubicSpline(t, data).derivative()(t)) < 1e-12
        if uniform:
            assert rel(ops.spline_calculus(t, data, "derivative", 2), CubicSpline(t, data).derivative(2)(t)) < 1e-10
        tp = np.linspace(t[0], t[-1], 1234)
        assert rel(ops.spline_calculus(t, data, "evaluate", tprime=tp), CubicSpline(t, data)(tp)) < 1e-13
        # antiderivatives (scri/waveform_base.py:697-703): exact integrals of the piecewise cubic, zero at t[0]
        assert rel(ops.spline_calculus(t, data, "antiderivative", 1), CubicSpline(t, data).antiderivative(1)(t)) < 1e-13
        assert rel(ops.spline_calculus(t, data, "antiderivative", 2), CubicSpline(t, data).antiderivative(2)(t)) < 1e-13
    # many tiles: the tile totals are carried across the tiles by 32 segments per column (spline_tile.cu: tile_scan_*)
    t, data = smooth_modes(n_times=20011, uniform=False, seed=22)
    data = data[:, :21] + 0.3                     # a non-zero mean, so that the running totals grow along the series
    for order in (1, 2):
        assert rel(ops.spline_calculus(t, data, "antiderivative", order), CubicSpline(t, data).antiderivative(order)(t)) < 1e-13
    # linear data is reproduced exactly (reference tests/test_waveform.py:183-270)
    t = np.linspace(-10.0, 100.0, 1000)
    lin = (np.arange(77) - 1j * np.arange(77))[None, :] * t[:, None]
    assert np.allclose(ops.spline_calculus(t, lin, "evaluate", tprime=t[5:-5] + 0.01), (np.arange(77) - 1j * np.arange(77))[None, :] * (t[5:-5] + 0.01)[:, None], rtol=1e-14)


def test_spline_strongly_nonuniform_steps():
    """Geometrically shrinking / growing steps slow the decay of the spline recurrences (up to 2/3 per row instead of
    0.27): scrib200_spline_prepare measures it and the tiles take a longer run-in.  Also the shortest series."""
    from scipy.interpolate import CubicSpline

    rng = np.random.default_rng(5)
    h = np.concatenate([0.1 * 0.9 ** np.arange(150), 0.1 * 0.9 ** 150 * 1.1 ** np.arange(200), np.full(300, 0.05) * rng.uniform(0.2, 1.8, 300)])
    t = np.concatenate([[0.0], np.cumsum(h)])
    data = np.exp(1j * np.outer(t, np.linspace(0.3, 2.0, 9))) * (1.0 + 0.1 * t[:, None])
    tp = np.sort(rng.uniform(t[0], t[-1], 3000))
    assert rel(ops.spline_calculus(t, data, "evaluate", tprime=tp), CubicSpline(t, data)(tp)) < 1e-13
    assert rel(ops.spline_calculus(t, data, "derivative", 1), CubicSpline(t, data).derivative()(t)) < 1e-12
    for n in (4, 5, 6, 17):
        tn = np.sort(rng.uniform(0.0, 1.0, n))
        dn = rng.normal(size=(n, 3)) + 1j * rng.normal(size=(n, 3))
        tpn = np.linspace(tn[0], tn[-1], 50)
        assert rel(ops.spline_calculus(tn, dn, "evaluate", tprime=tpn), CubicSpline(tn, dn)(tpn)) < 1e-12
        assert rel(ops.spline_calculus(tn, dn, "derivative", 1), CubicSpline(tn, dn).derivative()(tn)) < 1e-11


def test_boost_flux_and_eth_vs_oracle():
    """boost_flux (scri/flux.py:444-747, 27 expectation values in the reference) and apply_eth (waveform_modes.py:478-562)"""
    t, data = smooth_modes(n_times=300, seed=17)
    w = modes(t, data)
    Wo = R.Modes(t=t, data=data.copy())
    for ops_ in ("+", "-", "+-", "--", "-+"):
        assert rel(w.apply_eth(ops_), R.apply_eth(Wo, ops_)) < 1e-15
        assert rel(w.apply_eth(ops_, eth_convention="GHP"), R.apply_eth(Wo, ops_, "GHP")) < 1e-15
    assert np.array_equal(w.eth, w.apply_eth("+")) and np.array_equal(w.ethbar, w.apply_eth("-"))
    ref = R.boost_flux(Wo)
    assert rel(w.boost_flux(), ref) < 1e-11
    hd = w.copy()
    hd.dataType = sb.hdot
    hd.data = w.data_dot
    assert rel(w.boost_flux(hd), ref) < 1e-11
    E, p, J, B = w.poincare_fluxes()
    assert rel(B, ref) < 1e-11 and rel(E, R.energy_flux(Wo)) < 1e-12
    with pytest.raises(ValueError):
        hd.boost_flux()


def test_LLComparisonMatrix_vs_oracle():
    """scri/mode_calculations.py:106-206 (complex, not symmetrised; the reference's (y,y)/(y,z) accumulation included)"""
    t, d1 = smooth_modes(n_times=120, seed=51)
    _, d2 = smooth_modes(n_times=120, seed=52)
    w1, w2 = modes(t, d1), modes(t, d2)
    ref = R.LLComparisonMatrix(R.Modes(t=t, data=d1.copy()), R.Modes(t=t, data=d2.copy()))
    out = w1.LLComparisonMatrix(w2)
    assert out.shape == (120, 3, 3) and out.dtype == complex
    assert rel(out, ref) < 1e-13
    assert np.all(out[:, 1, 2] == 0)
    # with W1 = W2 the symmetrised real part of the well-formed elements is <LL>
    same = w1.LLComparisonMatrix(w1)
    LL = w1.LLMatrix()
    assert rel(same[:, 0, 0].real, LL[:, 0, 0]) < 1e-13 and rel(same[:, 2, 2].real, LL[:, 2, 2]) < 1e-13
    assert rel(0.5 * (same[:, 0, 1] + same[:, 1, 0]).real, LL[:, 0, 1]) < 1e-13


def test_dominant_eigenvector_and_angular_velocity_physics():
    """reference tests/test_mode_calculations.py:14-126 (simple cases)"""
    t = np.linspace(0.0, 20.0, 2001)
    omega = 0.3
    data = np.zeros((t.size, 21), complex)
    data[:, 4] = np.exp(-2j * omega * t)
    data[:, 0] = np.exp(2j * omega * t)
    w = modes(t, data, ell_max=4)
    assert np.allclose(w.LLDominantEigenvector(), np.array([0, 0, 1.0])[None, :], atol=1e-14)
    assert np.allclose(w.angular_velocity()[5:-5], np.array([0, 0, omega])[None, :], atol=1e-9)
    Rq = quat.normalized(np.array([1.0, 2.0, 3.0, 4.0]))
    w.rotate_decomposition_basis(Rq)
    expect = quat.rotate_vector(quat.conj(Rq), np.array([0, 0, omega]))
    assert np.allclose(w.angular_velocity()[5:-5], expect[None, :], atol=1e-9)
    zhat = quat.rotate_vector(quat.conj(Rq), np.array([0, 0, 1.0]))
    dpa = w.LLDominantEigenvector(RoughDirection=zhat)
    assert np.allclose(dpa, zhat[None, :], atol=1e-13)


def test_corotating_frame_round_trip():
    """config 1 (shortened): to_corotating_frame then to_inertial_frame restores the modes
    (reference tests/test_mode_calculations.py:75-126 tolerance 1e-8)."""
    w = sb.sample_waveforms.fake_precessing_waveform(t_1=400.0)
    ref = w.data.copy()
    w.to_corotating_frame()
    assert w.frameType == sb.Corotating and w.frame.shape == (w.n_times, 4)
    # in the corotating frame the modes vary slowly: time derivative norm drops by orders of magnitude
    assert np.median(np.sum(abs(w.data_dot) ** 2, 1)) < 1e-2 * np.median(np.sum(abs(ops.spline_calculus(w.t, ref, "derivative", 1)) ** 2, 1))
    w.to_inertial_frame()
    assert w.frameType == sb.Inertial
    assert np.allclose(w.data, ref, rtol=0, atol=1e-12)


@pytest.mark.parametrize("same", [True, False])
@pytest.mark.parametrize("width,cplx", [(1, False), (2, True), (3, False), (4, True), (6, False)])
def test_sparse_expectation_every_kernel_against_dense(same, width, cplx, monkeypatch):
    """<a|M_k|b>(t) (scri/flux.py:40-78) for random banded matrices through every kernel the product can pick: lanes along
    time (real / complex values, one array / two arrays, 1..4 entries per column, a column block count above one), the
    warp-per-step ELL and COO kernels (forced by SCRIB200_EXPECTATION_WARP, or chosen for 6 entries per column), against the
    dense contraction.  Columns without entries, matrices of different widths and 5 matrices (two launches of <= 4) included."""
    rng = np.random.default_rng(100 * width + 10 * cplx + same)
    n, N, K = 285, 333, 5
    a = rng.normal(size=(N, n)) + 1j * rng.normal(size=(N, n))
    b = a if same else rng.normal(size=(N, n)) + 1j * rng.normal(size=(N, n))
    mats, dense = [], []
    for k in range(K):
        wk = width if k != 1 else max(1, width - 1)            # one narrower matrix: its slots are padded
        rows, cols, vals = [], [], []
        for c in range(n):
            if c % 17 == 5:                                     # columns without entries
                continue
            r = np.unique(np.clip(c + rng.integers(-35, 36, size=wk), 0, n - 1))
            v = rng.normal(size=r.size) + (1j * rng.normal(size=r.size) if cplx else 0.0)
            rows += list(r)
            cols += [c] * r.size
            vals += list(v)
        M = np.zeros((n, n), dtype=complex)
        M[rows, cols] = vals
        dense.append(M)
        mats.append((np.array(rows), np.array(cols), np.array(vals, dtype=complex if cplx else float)))
    want = np.stack([np.einsum("tr,rc,tc->t", a.conj(), M, b) for M in dense], axis=1)
    got = ops.sparse_expectation(a, b, mats)
    assert rel(got, want) < 1e-13
    monkeypatch.setenv("SCRIB200_EXPECTATION_WARP", "1")
    ops._sparse_cache.clear()
    assert rel(ops.sparse_expectation(a, b, mats), want) < 1e-13
    ops._sparse_cache.clear()


def test_full_size_fluxes_config5_slice():
    """l<=16 fluxes on 1e5 steps (a slice of config 5): linearity / scaling properties + oracle on a window."""
    N = 100_000
    t, data = smooth_modes(n_times=N, ell_max=16, t0=0.0, t1=1e4, seed=31)
    w = modes(t, data, ell_max=16)
    E, p, J, Bst = w.poincare_fluxes()
    w2 = modes(t, 2.0 * data, ell_max=16)
    E2, p2, J2, Bst2 = w2.poincare_fluxes()
    assert np.allclose(Bst2, 4 * Bst, rtol=1e-11, atol=1e-12 * abs(Bst).max())
    assert np.allclose(E2, 4 * E, rtol=1e-13) and np.allclose(p2, 4 * p, rtol=1e-12, atol=1e-14) and np.allclose(J2, 4 * J, rtol=1e-12, atol=1e-14)
    assert (E >= 0).all()
    lo, hi = 40_000, 41_000
    Wo = R.Modes(t=t[lo:hi], data=data[lo:hi].copy(), ell_min=2, ell_max=16)
    assert rel(E[lo + 200 : hi - 200], R.energy_flux(Wo)[200:-200]) < 1e-11
    assert rel(p[lo + 200 : hi - 200], R.momentum_flux(Wo)[200:-200]) < 1e-11
    assert rel(J[lo + 200 : hi - 200], R.angular_momentum_flux(Wo)[200:-200]) < 1e-11


# ------------------------------------------------------------------ AsymptoticBondiData, grid_multiply (a23, a24)
def _random_abd(ell_max=4, n_times=240, seed=11):
    from oracle import abd_ref as A

    rng = np.random.default_rng(seed)
    u = np.linspace(-10.0, 30.0, n_times)
    n = (ell_max + 1) ** 2
    data = {}
    for name, s in A.SPINS.items():
        c = rng.normal(size=n) + 1j * rng.normal(size=n)
        w = rng.uniform(0.05, 0.5, size=n)
        d = 0.1 * c[None, :] * np.exp(1j * w[None, :] * u[:, None])
        d[:, : s * s] = 0.0                                   # no modes below |s|
        data[name] = d
    mine = sb.AsymptoticBondiData(u, ell_max)
    for name in A.FIELDS:
        setattr(mine, name, data[name])
    return mine, A.ABD(u, ell_max, {k: v.copy() for k, v in data.items()})


@pytest.mark.parametrize("kw", [
    dict(supertranslation=real_supertranslation(2, seed=9), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03]),
    dict(boost_velocity=[0.0, 0.05, -0.02]),
    dict(time_translation=1.5, frame_rotation=[0.3, -0.4, 0.5, 0.7]),
    dict(space_translation=np.array([0.1, -0.2, 0.3]), output_ell_max=3, working_ell_max=9),
])
def test_abd_transform_vs_oracle(kw):
    """All six fields through scri/asymptotic_bondi_data/transformations.py:199-431 (Horner ladders in eth u'/k)."""
    from oracle import abd_ref as A

    mine, ref = _random_abd()
    out = mine.transform(**kw)
    exp = A.transform(ref, **kw)
    assert np.array_equal(out.u, exp.u)                       # output time grid: bit-exact ((u - dt) / gamma, masked)
    assert out.ell_max == exp.ell_max
    for name in A.FIELDS:
        assert rel(getattr(out, name).ndarray, exp.data[name]) < RTOL, name


def test_abd_schwarzschild_boost_and_charges():
    """reference tests/test_asymptoticbondidata.py:96-117 on the GPU path"""
    import math

    mass, ell_max = 1.0, 4
    u = np.linspace(0, 100, num=200)
    abd = sb.AsymptoticBondiData(u, ell_max)
    psi2 = np.zeros((ell_max + 1) ** 2, complex)
    psi2[0] = -mass * math.sqrt(4 * math.pi)
    abd.psi2 = psi2
    assert np.allclose(abd.bondi_rest_mass(), mass, atol=1e-14)
    for v in [np.array([0.1, 0.0, 0.0]), np.array([0.0, 0.1, 0.0]), np.array([0.0, 0.0, 0.1])]:
        gamma = 1 / np.sqrt(1 - v @ v)
        abdprime = abd.transform(boost_velocity=v)
        assert np.allclose(abdprime.bondi_four_momentum(), mass * gamma * np.array([1, *-v]), atol=1e-13, rtol=1e-13)
        assert np.allclose(abdprime.bondi_rest_mass(), mass, atol=1e-13)


def test_grid_multiply_and_modes_time_series_vs_oracle():
    """scri/modes_time_series.py:72-202"""
    from oracle import abd_ref as A
    from scipy.interpolate import CubicSpline

    mine, ref = _random_abd(ell_max=5, n_times=150, seed=3)
    sig, p3 = mine.sigma, mine.psi3
    prod = sig.grid_multiply(p3)
    assert prod.spin_weight == 1 and prod.ell_max == 5
    assert rel(prod.ndarray, A.grid_multiply(ref.data["sigma"], 2, ref.data["psi3"], -1)) < RTOL
    prod2 = sig.grid_multiply(sig.bar, working_ell_max=12, output_ell_max=7)
    assert prod2.spin_weight == 0 and prod2.ell_max == 7
    assert rel(prod2.ndarray, A.grid_multiply(ref.data["sigma"], 2, A.modes_bar(ref.data["sigma"], 2), -2, working_ell_max=12, output_ell_max=7)) < RTOL
    assert rel(sig.bar.ndarray, A.modes_bar(ref.data["sigma"], 2)) == 0.0
    assert rel(sig.dot.ndarray, CubicSpline(ref.u, ref.data["sigma"]).derivative()(ref.u)) < 1e-11
    assert rel(sig.int.ndarray, CubicSpline(ref.u, ref.data["sigma"]).antiderivative()(ref.u)) < 1e-12
    tn = np.linspace(ref.u[3], ref.u[-3], 77)
    assert rel(mine.interpolate(tn).psi1.ndarray, CubicSpline(ref.u, ref.data["psi1"])(tn)) < 1e-12
    assert rel(mine.psi2.eth_GHP.ndarray, A.modes_eth(ref.data["psi2"], 0) / np.sqrt(2)) < 1e-15
    # salm2map alone against the restated spinsfast
    from oracle import spinsfast as ospf

    g = ops.salm2map(ref.data["psi3"][:20], -1, 5, 13, 13)
    assert rel(g, ospf.salm2map(ref.data["psi3"][:20], -1, 5, 13, 13)) < 1e-13


def test_config4_sized_swsh_round_trip_and_products():
    """BASELINE config 4 in miniature: l <= 32 fields on the 129 x 129 grid (the dense synthesis GEMM with K = 2178 and the
    large-grid analysis path): salm2map -> map2salm is the identity on band-limited data for every spin, and
    grid_multiply reproduces the exact product of low-l factors whatever the working band limit."""
    rng = np.random.default_rng(8)
    N, L = 24, 32
    for s in (0, -2, 1):
        a = rng.normal(size=(N, (L + 1) ** 2)) + 1j * rng.normal(size=(N, (L + 1) ** 2))
        a[:, : s * s] = 0.0
        g = ops.salm2map(a, s, L, 2 * L + 1, 2 * L + 1)
        assert g.shape == (N, 65, 65)
        back = ops.map2salm(g, s, L)
        assert rel(back, a) < 1e-12
        g2 = ops.salm2map(a, s, L, 129, 129)
        back2 = ops.map2salm(g2, s, L, 129, 129)
        assert rel(back2, a) < 1e-12
    # product of two fields computed on two different working grids agrees (no aliasing once L_w >= l1 + l2)
    t = np.linspace(0.0, 1.0, N)
    f = sb.ModesTimeSeries(rng.normal(size=(N, 17 * 17)) + 1j * rng.normal(size=(N, 17 * 17)), t, 0)
    h = rng.normal(size=(N, 17 * 17)) + 1j * rng.normal(size=(N, 17 * 17))
    h[:, :4] = 0.0
    h = sb.ModesTimeSeries(h, t, -2)
    p1 = f.grid_multiply(h, working_ell_max=32, output_ell_max=32)
    p2 = f.grid_multiply(h, working_ell_max=64, output_ell_max=32)
    assert p1.spin_weight == -2 and p1.ell_max == 32
    assert rel(p1.ndarray, p2.ndarray) < 1e-12


def test_batched_transform_equals_single_transforms():
    """BASELINE config 3 in miniature: a batch of waveforms sharing the time axis and the transformation goes through
    one synthesis, one spline (batch in gridDim.z) and one analysis launch and equals the per-waveform results bit for bit."""
    import torch

    B, N = 5, 333
    t = np.linspace(0.0, 60.0, N)
    batch = np.stack([smooth_modes(n_times=N, t0=0.0, t1=60.0, seed=70 + b)[1] for b in range(B)])
    pl = P.TransformPlan(2, 8, sb.h, **BMS)
    td, bd = ops.to_device(t), ops.to_device(batch)
    up, out = pl.run_batch(td, bd)
    assert out.shape[0] == B and out.shape[1] == up.shape[0]
    for b in range(B):
        up1, out1 = pl.run(td, bd[b].contiguous())
        assert torch.equal(up1, up) and torch.equal(out1, out[b])
    ref = R.transform(R.Modes(t=t, data=batch[3].copy()), **BMS)
    assert rel(out[3].cpu().numpy(), ref.data) < RTOL
    from scri_b200 import parallel

    up2, out2 = parallel.transform_batch(pl, td, bd)
    assert torch.equal(out2, out)
    # the second call on the same time-axis tensor assumes its retained block; a time axis rewritten IN PLACE (same storage,
    # other retained block) must be noticed and the call repeated unassumed; host blocks through one shared preparation
    up3, out3 = pl.run_batch(td, bd)
    assert torch.equal(up3, up) and torch.equal(out3, out)
    t_new = np.linspace(0.0, 25.0, N)          # a finer axis: another retained block under the same supertranslation
    td.copy_(torch.from_numpy(t_new).to(td.device))
    up4, out4 = pl.run_batch(td, bd)
    fresh = P.TransformPlan(2, 8, sb.h, **BMS)
    up5, out5 = fresh.run_batch(ops.to_device(t_new), bd)
    assert torch.equal(up4, up5)
    assert torch.equal(out4, out5)
    assert up4.shape[0] != up.shape[0] or not torch.equal(up4, up)
    uh, mh = parallel.transform_batch_host(fresh, t_new, batch, sub_batch=2)
    assert np.array_equal(uh, up5.cpu().numpy()) and np.array_equal(mh, out5.cpu().numpy())


def test_million_step_transform_window_vs_oracle():
    """Largest size of BASELINE.json (1e6 time steps): 4167 time tiles, 10 GB of intermediates, 64-bit indexing.  The
    spline couples samples only locally, so a 3000-sample window of the input reproduces the interior of the full result."""
    N = 1_000_000
    t = np.linspace(0.0, 1e5, N)
    _, data = smooth_modes(n_times=N, t0=0.0, t1=1e5, seed=16)
    kw = dict(supertranslation=real_supertranslation(3, seed=2), frame_rotation=[1.0, -2.0, 0.5, 3.0])     # no boost: the window stays put
    pl = P.TransformPlan(2, 8, sb.h, **kw)
    up, out = pl.run(ops.to_device(t), ops.to_device(data))
    upn, outn = up.cpu().numpy(), out.cpu().numpy()
    assert upn.shape[0] > N - 10 and np.all(np.diff(upn) > 0)
    for lo in (0, 499_000, N - 3000):
        ref = R.transform(R.Modes(t=t[lo : lo + 3000], data=data[lo : lo + 3000].copy()), **kw)
        inner = ref.t[200:-200]
        sel = np.searchsorted(upn, inner)
        assert np.array_equal(upn[sel], inner)
        assert rel(outn[sel], ref.data[200:-200]) < RTOL


def _sharded_flux_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist

    from scri_b200 import parallel

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)     # one GPU here: gloo carries the halos (NCCL on a real node)
    try:
        t, data = smooth_modes(n_times=4000, t0=0.0, t1=400.0, seed=23)
        lo, hi = parallel.shard_range(t.size, rank, world)
        td, dd = ops.to_device(t[lo:hi].copy()), ops.to_device(data[lo:hi].copy())
        e, p, j = parallel.sharded_fluxes(td, dd, 2, 8)
        d2 = parallel.sharded_time_derivative(td, dd, 2)
        q.put((rank, lo, hi, e.cpu().numpy(), p.cpu().numpy(), j.cpu().numpy(), d2.cpu().numpy()))
    finally:
        dist.destroy_process_group()


def test_time_sharded_fluxes_world2():
    """SURVEY 8(e): time sharding - halo exchange of input modes, local spline derivative, pointwise fluxes - equals the
    single-process result (two ranks sharing the one GPU of the test box, gloo for the halos)."""
    import socket

    import torch.multiprocessing as mp

    s_ = socket.socket()
    s_.bind(("127.0.0.1", 0))
    port = s_.getsockname()[1]
    s_.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_flux_worker, args=(r, 2, port, q)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = sorted([q.get(timeout=300) for _ in range(2)], key=lambda x: x[0])
    for pr in procs:
        pr.join(timeout=60)
    t, data = smooth_modes(n_times=4000, t0=0.0, t1=400.0, seed=23)
    w = modes(t, data)
    E, pd, J = w.energy_flux(), w.momentum_flux(), w.angular_momentum_flux()
    dd = w.data_ddot
    assert (res[0][1], res[0][2], res[1][2]) == (0, 2000, 4000)
    assert rel(np.concatenate([r[3] for r in res]), E) < 1e-12
    assert rel(np.concatenate([r[4] for r in res]), pd) < 1e-12
    assert rel(np.concatenate([r[5] for r in res]), J) < 1e-12
    assert rel(np.concatenate([r[6] for r in res]), dd) < 1e-10


@pytest.mark.parametrize("grid", [dict(n_theta=27, n_phi=31), dict(n_theta=33, n_phi=25), dict(n_theta=26, n_phi=26, ell_max=5),
                                  dict(ell_max=9), dict(ell_max=10), dict(ell_max=12), dict(n_theta=67, n_phi=19),
                                  dict(n_theta=19, n_phi=19, ell_max=9), dict(n_theta=31, n_phi=31, ell_max=15)])
def test_transform_on_user_chosen_grids(grid):
    """`n_theta`, `n_phi` and the output `ell_max` are user keywords (scri/waveform_grid.py:97-110, 627): non-square and
    oversampled grids take the general analysis path (quadrature tables and tile sizes follow the grid).  With the
    supertranslation of BMS the default grid is 25 x 25; the output band limits 9 .. 12 on it and the grids added with them
    run the non-aliased tiled analysis at time tiles 4 and 2, the aliased one at 2 (67 x 19, also the spline remap's
    two-step time tile), the persistent tensor-core kernel with two m-blocks (19 x 19, ell_max 9) and the time-major fused
    kernel (31 x 31, ell_max 15), all through the oracle comparison.  ell_max = 15 needs the larger grid: on 25 rings the
    quadrature integrand reaches past n_theta - 2, where this quadrature and the oracle's torus extension alias
    differently (2e-12 apart even in long double)."""
    t, data = smooth_modes(n_times=300, seed=12)
    kw = dict(BMS, **grid)
    out = modes(t, data).transform(**kw)
    ref = R.transform(R.Modes(t=t, data=data.copy()), **kw)
    assert np.array_equal(out.t, ref.t)
    assert out.ell_max == grid.get("ell_max", 8) and out.data.shape == ref.data.shape
    assert rel(out.data, ref.data) < RTOL
    g = modes(t, data).to_grid(**{k: v for k, v in kw.items() if k != "ell_max"})
    go = R.from_modes(R.Modes(t=t, data=data.copy()), **{k: v for k, v in kw.items() if k != "ell_max"})
    assert (g.n_theta, g.n_phi) == (go.n_theta, go.n_phi) and rel(g.data, go.data) < RTOL


def _rand_modes(rng, N, L, s, ell_min=0):
    a = rng.normal(size=(N, (L + 1) ** 2)) + 1j * rng.normal(size=(N, (L + 1) ** 2))
    a[:, : s * s] = 0.0
    return a[:, ell_min**2 :]


@pytest.mark.parametrize("case", [(2, 3, -2, 4, None, None, 6), (0, 4, 1, 2, None, 6, 1), (2, 5, -2, 5, 6, 4, 9), (-1, 3, 0, 3, 3, 3, 4),
                                  (2, 8, -2, 8, None, 8, 37), (0, 12, 2, 8, None, 20, 10)])
def test_fused_modes_product_vs_oracle(case):
    """K9 (scrib200_modes_product) against the oracle's grid_multiply (scri/modes_time_series.py:142-202): default and
    aliased working grids, ragged time counts (the kernel walks 4 steps at a time), output band limits above and below
    the factors'."""
    from oracle import abd_ref as A

    s1, L1, s2, L2, Lw, Lo, N = case
    rng = np.random.default_rng(21)
    a, b = _rand_modes(rng, N, L1, s1), _rand_modes(rng, N, L2, s2)
    ref = A.grid_multiply(a, s1, b, s2, working_ell_max=Lw, output_ell_max=Lo)
    n = 2 * (L1 + L2 if Lw is None else Lw) + 1
    out = ops.modes_product(a, s1, 0, L1, b, s2, 0, L2, n, n, L1 if Lo is None else Lo)
    assert out is not None and out.shape == ref.shape
    assert rel(out, ref) < RTOL
    for shape in (0, 1, 2):   # 16 warps x 5 M, 8 warps x 9 M, CTA pairs (thread-block cluster, distributed shared memory)
        assert rel(ops.modes_product(a, s1, 0, L1, b, s2, 0, L2, n, n, L1 if Lo is None else Lo, shape=shape), ref) < RTOL


def test_fused_modes_product_ell_min_and_3j_multiply():
    """A factor stored from ell_min = 2 (as WaveformModes data is) and ModesTimeSeries.multiply against the 3j sums of
    spherical_functions' Modes.multiply (oracle.sf.modes_multiply; bms_charges.py:40-187)."""
    from oracle import abd_ref as A, sf as osf

    rng = np.random.default_rng(22)
    N = 11
    a0, b = _rand_modes(rng, N, 5, 2), _rand_modes(rng, N, 4, -1)
    out = ops.modes_product(a0[:, 4:], 2, 2, 5, b, -1, 0, 4, 19, 19, 5)
    assert rel(out, A.grid_multiply(a0, 2, b, -1)) < RTOL
    t = np.linspace(0.0, 1.0, N)
    f, g = sb.ModesTimeSeries(a0, t, 2), sb.ModesTimeSeries(b, t, -1)
    for trunc, Lo in ((max, 5), (sum, 9), (lambda tup: 3, 3), (lambda tup: 12, 12)):
        p = f.multiply(g, truncator=trunc)
        assert p.spin_weight == 1 and p.ell_max == Lo
        assert rel(p.ndarray, osf.modes_multiply(a0, 2, 5, b, -1, 4, Lo)) < RTOL


def test_fused_modes_product_config4_size_equals_dense_path():
    """BASELINE config 4 size (ell <= 32 factors, 129 x 129 working grid): the fused separable kernel against the dense
    synthesis GEMM -> product -> analysis chain of the same library, and linearity in each factor."""
    rng = np.random.default_rng(23)
    N, L = 10, 32
    a, b = _rand_modes(rng, N, L, 2), _rand_modes(rng, N, L, -2)
    fused = ops.grid_multiply(a, 2, 0, L, b, -2, 0, L, 129, 129, 64, output_ell_max=32)
    dense = ops.grid_multiply(a, 2, 0, L, b, -2, 0, L, 129, 129, 64, output_ell_max=32, fused=False)
    assert fused.shape == dense.shape == (N, 33 * 33)
    assert rel(fused, dense) < RTOL
    from oracle import abd_ref as A   # the reference's chain itself on two steps (a few seconds of CPU at this size)

    assert rel(fused[:2], A.grid_multiply(a[:2], 2, b[:2], -2, working_ell_max=64, output_ell_max=32)) < RTOL
    for shape in (0, 1, 2):   # the instantiated kernel shapes (16 warps x 5 M, 8 warps x 9 M, CTA pairs)
        assert rel(ops.modes_product(a, 2, 0, L, b, -2, 0, L, 129, 129, 32, shape=shape), dense) < RTOL
    a2 = _rand_modes(rng, N, L, 2)
    lin = ops.grid_multiply(a + 0.5 * a2, 2, 0, L, b, -2, 0, L, 129, 129, 64, output_ell_max=32)
    assert rel(lin, fused + 0.5 * ops.grid_multiply(a2, 2, 0, L, b, -2, 0, L, 129, 129, 64, output_ell_max=32)) < RTOL


@pytest.mark.parametrize("case", [(-2, 0, 8, 17, 17, 5), (2, 2, 12, 25, 25, 9), (1, 0, 16, 40, 37, 4), (0, 0, 32, 65, 65, 6), (-1, 0, 32, 129, 129, 3)])
def test_separable_salm2map_vs_dense_and_oracle(case):
    """The separable synthesis on spinsfast's regular grid (scrib200_theta_synth + the phi-DFT GEMM) against the dense
    synthesis GEMM of the same library and, at the small sizes, against the restated spinsfast.salm2map
    (scri/modes_time_series.py:177-182): spins, ell_min > 0, rectangular and oversampled grids, ragged time counts."""
    from oracle import spinsfast as ospf

    s, lmin, L, nth, nph, N = case
    rng = np.random.default_rng(31)
    a = _rand_modes(rng, N, L, s, ell_min=lmin)
    sep = ops.salm2map(a, s, L, nth, nph, ell_min=lmin, separable=True)
    dense = ops.salm2map(a, s, L, nth, nph, ell_min=lmin, separable=False)
    assert sep.shape == dense.shape == (N, nth, nph)
    assert rel(sep, dense) < 1e-13
    if L <= 16:
        full = np.zeros((N, (L + 1) ** 2), dtype=complex)
        full[:, lmin**2 :] = a
        assert rel(sep, ospf.salm2map(full, s, L, nth, nph)) < 1e-13


@pytest.mark.parametrize("case", [(-2, 0, 8, 17, 17, 5), (2, 2, 12, 25, 25, 9), (1, 0, 16, 40, 37, 4), (0, 0, 32, 65, 65, 6), (-1, 1, 32, 129, 129, 3)])
def test_separable_map2salm_vs_smem_kernels_and_oracle(case):
    """The separable analysis (phi-DFT GEMM + scrib200_theta_quad) against the shared-memory kernels of
    scrib200_map2salm and the restated spinsfast.map2salm (scri/waveform_grid.py:303-307), on maps that are NOT band
    limited (white noise on the grid: the quadrature itself is compared, not a round trip) and on a round trip."""
    from oracle import spinsfast as ospf

    s, lmin, L, nth, nph, N = case
    rng = np.random.default_rng(32)
    f = rng.normal(size=(N, nth, nph)) + 1j * rng.normal(size=(N, nth, nph))
    sep = ops.map2salm(f, s, L, nth, nph, ell_min=lmin, separable=True)
    old = ops.map2salm(f, s, L, nth, nph, ell_min=lmin, separable=False)
    assert sep.shape == old.shape == (N, (L + 1) ** 2 - lmin**2)
    assert rel(sep, old) < 1e-13
    if L <= 16:
        assert rel(sep, ospf.map2salm(f, s, L)[:, lmin**2 :]) < 1e-13
    a = _rand_modes(rng, N, L, s, ell_min=lmin)
    back = ops.map2salm(ops.salm2map(a, s, L, nth, nph, ell_min=lmin, separable=True), s, L, nth, nph, ell_min=lmin, separable=True)
    assert rel(back, a) < RTOL


def test_transform_large_band_limit_vs_oracle():
    """A transform at ell_max = 20 (working grid 49 x 49: beyond the shared-memory tile kernels of the analysis, which
    then runs separable on the tensor cores) against the oracle, and its inverse round trip."""
    t, data = smooth_modes(n_times=160, ell_max=20, seed=14)
    out = modes(t, data, ell_max=20).transform(**BMS)
    ref = R.transform(R.Modes(t=t, data=data.copy(), ell_max=20), **BMS)
    assert np.array_equal(out.t, ref.t) and out.data.shape == ref.data.shape
    assert rel(out.data, ref.data) < RTOL


def _sharded_transform_worker(rank, world, port, q, kw, n_times, t1):
    import torch
    import torch.distributed as dist

    from scri_b200 import parallel

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)     # one GPU here: gloo carries the halos (NCCL on a real node)
    try:
        t, data = smooth_modes(n_times=n_times, t0=0.0, t1=t1, seed=29)
        lo, hi = parallel.shard_range(t.size, rank, world)
        td, dd = ops.to_device(t[lo:hi].copy()), ops.to_device(data[lo:hi].copy())
        plan = P.TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **kw)
        try:
            u, m = parallel.sharded_transform(plan, td, dd)
            q.put((rank, u.cpu().numpy(), m.cpu().numpy(), None))
        except ValueError as e:
            q.put((rank, None, None, str(e)))
    finally:
        dist.destroy_process_group()


def _run_sharded_transform(kw, n_times, t1, world=2):
    import socket

    import torch.multiprocessing as mp

    s_ = socket.socket()
    s_.bind(("127.0.0.1", 0))
    port = s_.getsockname()[1]
    s_.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_transform_worker, args=(r, world, port, q, kw, n_times, t1)) for r in range(world)]
    for pr in procs:
        pr.start()
    res = sorted([q.get(timeout=300) for _ in range(world)], key=lambda x: x[0])
    for pr in procs:
        pr.join(timeout=60)
    return res


def test_time_sharded_transform_world2():
    """SURVEY 8(e): one series sharded by time over two ranks - halo exchange of the input modes, local synthesis /
    splines / analysis, outputs owned by the rank that owns the input sample - against the single-process transform:
    output times bit-exact, modes to 1e-12.  A supertranslation + rotation needs a fixed halo; a boost over a short series
    still fits; a boost that moves the input window by more than a block is refused with the reason."""
    for kw, n_times, t1 in (
        (dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0]), 6000, 600.0),
        (dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0], boost_velocity=[0.01, 0.02, 0.03]), 4000, 100.0),
    ):
        res = _run_sharded_transform(kw, n_times, t1)
        assert all(r[3] is None for r in res), res[0][3]
        t, data = smooth_modes(n_times=n_times, t0=0.0, t1=t1, seed=29)
        ref = modes(t, data).transform(**kw)
        u = np.concatenate([r[1] for r in res])
        m = np.concatenate([r[2] for r in res])
        assert np.array_equal(u, ref.t)
        assert rel(m, ref.data) < RTOL
    res = _run_sharded_transform(dict(boost_velocity=[0.3, 0.4, 0.5]), 4000, 400.0)    # drift ~ 0.7 N samples: more than a block
    assert all(r[3] is not None and "shard by waveform" in r[3] for r in res)


@pytest.mark.parametrize("n_slabs", [3, 8])
def test_streaming_end_to_end_pipeline_is_bitwise_identical(n_slabs):
    """WaveformGrid.transform's host path: input slabs synthesized as they land, output slabs remapped / analysed / copied back
    as soon as their input window is there (TransformPlan._run_streaming).  The grid array is poisoned with NaN first, so
    an output computed from a row that was not synthesized yet could not go unnoticed; the result equals the single-launch
    device path bit for bit, with and without a boost."""
    for kw in (BMS, dict(supertranslation=real_supertranslation(4), frame_rotation=[1.0, 2.0, 3.0, 4.0])):
        t, data = smooth_modes(n_times=12000, t0=0.0, t1=1200.0, seed=41)
        plan = P.TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **kw)
        td = ops.to_device(t)
        u1, m1 = plan.run(td, ops.to_device(data))
        a_d, slabs, fut = ops.to_device_slabs(data, np.complex128, n_slabs=n_slabs)
        u2, m2 = plan._run_streaming(td, a_d, slabs, t, debug_poison=True)
        fut.result()
        assert np.array_equal(u2, u1.cpu().numpy())
        assert np.isfinite(m2).all() and np.array_equal(m2, m1.cpu().numpy())
    out = modes(t, data).transform(**BMS)          # the public call takes the same path
    ref = R.transform(R.Modes(t=t, data=data.copy()), **BMS)
    assert np.array_equal(out.t, ref.t) and rel(out.data, ref.data) < RTOL


def test_interpolate_data_and_frame():
    """WaveformBase.interpolate (scri/waveform_base.py:949-967; reference tests/test_waveform.py:205-260): data through the
    not-a-knot cubic spline of every column (scipy's CubicSpline is the reference's own call), frame through squad; a
    constant waveform is reproduced to the reference's 4.5e-16."""
    from scipy.interpolate import CubicSpline

    from scri_b200 import _quaternion as Q

    t, data = smooth_modes(n_times=700, t0=0.0, t1=70.0, seed=51, uniform=False)
    ang = 0.3 * t + 0.05 * np.sin(t)
    frame = Q.qexp_vec(0.5 * ang[:, None] * np.array([0.1, -0.2, 0.97])[None, :])
    w = modes(t, data, frameType=sb.Corotating, frame=frame)
    t_out = (t[:-1] + t[1:]) / 2.0
    w_out = w.interpolate(t_out)
    assert w.ensure_validity(alter=False) and w_out.ensure_validity(alter=False)
    assert w_out.frameType == sb.Corotating and w_out.dataType == sb.h and w_out.r_is_scaled_out and w_out.m_is_scaled_out
    assert w_out.num != w.num and np.all(w_out.t == t_out) and np.all(w_out.LM == w.LM)
    assert w_out.data.shape == (len(t_out), w.n_modes)
    assert np.array_equal(w_out.frame, Q.squad(frame, t, t_out))
    assert rel(w_out.data, CubicSpline(t, data)(t_out)) < RTOL
    assert np.array_equal(w.data, data)                         # the input is untouched
    const = modes(t, np.tile(data[:1], (t.size, 1)), frameType=sb.Corotating, frame=np.tile(frame[:1], (t.size, 1)))
    c_out = const.interpolate(t_out)
    assert np.abs(c_out.data - data[:1]).max() <= 4.5e-16 * np.abs(data[:1]).max() * 4
    assert np.abs(c_out.frame - frame[:1]).max() <= 4.5e-16


def test_align_decomposition_frame_to_modes_and_slicing():
    """scri/rotations.py:114-265 and scri/waveform_modes.py:953-1021: after the alignment the dominant eigenvector of <LL>
    at the fiducial time is the z axis of the decomposition frame, the (2, +-2) phases agree, the x axis is on nHat's side,
    and the waveform still is the same physical waveform (back in the inertial frame it equals the original)."""
    import math

    w0 = sb.sample_waveforms.fake_precessing_waveform(t_0=-20.0, t_1=300.0, dt=0.1, ell_max=4)
    ref = w0.data.copy()
    w = w0.copy().to_corotating_frame()
    t_fid = 123.456
    sub = w[100:140, 2:4]
    assert sub.ells == (2, 3) and sub.data.shape == (40, 12) and sub.frame.shape == (40, 4) and np.array_equal(sub.t, w.t[100:140])
    assert np.array_equal(sub.data, w.data[100:140, :12])
    with pytest.raises(ValueError):
        w0.copy().align_decomposition_frame_to_modes(t_fid)      # inertial frame: refused, as in the reference
    w.align_decomposition_frame_to_modes(t_fid)
    i = int(np.searchsorted(w.t, t_fid))
    inst = w[i - 6 : i + 6].interpolate(np.array([t_fid]))
    V = inst.LLDominantEigenvector()[0]
    assert abs(abs(V[2]) - 1.0) < 1e-9 and np.hypot(V[0], V[1]) < 1e-4
    a22, a2m2 = inst.data[0, inst.index(2, 2)], inst.data[0, inst.index(2, -2)]
    dphi = math.atan2(a22.imag, a22.real) - math.atan2(a2m2.imag, a2m2.real)
    assert abs(math.remainder(dphi, 2 * math.pi)) < 1e-6
    from scri_b200 import _quaternion as Q

    xq = np.array([0.0, 1.0, 0.0, 0.0])
    assert Q.qmul(Q.qmul(inst.frame[0], xq), Q.qinverse(inst.frame[0]))[1] > 0      # x axis on the side of nHat = x
    back = w.copy().to_inertial_frame()
    assert rel(back.data, ref) < 1e-10


def test_bms_charges_vs_3j_oracle():
    """scri/asymptotic_bondi_data/bms_charges.py:77-269 on the GPU path (every product through the fused kernel K9) against the
    oracle, whose products are the literal 3j sums of spherical_functions' Modes.multiply: four-momentum, angular momentum,
    boost and centre-of-mass charges, dimensionless spin, the four supermomentum definitions."""
    from oracle import abd_ref as A

    mine, ref = _random_abd(ell_max=4, n_times=120, seed=61)
    ref.data["psi2"][:, 0] += -10.0 * np.sqrt(4 * np.pi)         # a mass monopole: the four-momentum is timelike
    mine.psi2 = ref.data["psi2"]
    P, J, N, G = A.bms_charges(ref)
    assert rel(mine.bondi_four_momentum(), P) < RTOL
    assert rel(mine.bondi_angular_momentum(), J) < RTOL
    assert rel(mine.bondi_boost_charge(), N) < 1e-11
    assert rel(mine.bondi_CoM_charge(), G) < RTOL
    M2 = (P[:, 0] ** 2 - np.sum(P[:, 1:] ** 2, axis=1))[:, None]
    v = P[:, 1:] / P[:, :1]
    vn = np.linalg.norm(v, axis=1)[:, None]
    gam = 1 / np.sqrt(1 - vn**2)
    chi = (gam * (J + np.cross(v, N)) - (gam - 1) * np.sum(J * v / vn, axis=1)[:, None] * v / vn) / M2
    assert rel(mine.bondi_dimensionless_spin(), chi) < 1e-10
    for kind, short in (("Bondi-Sachs", "bs"), ("Moreschi", "m"), ("G", "g"), ("geroch-winicour", "gw")):
        assert rel(mine.supermomentum(kind).ndarray, A.supermomentum(ref, short)) < RTOL
    assert rel(mine.supermomentum("M", integrated=True, working_ell_max=10).ndarray, A.supermomentum(ref, "m", working_ell_max=10, integrated=True)) < RTOL
    with pytest.raises(ValueError):
        mine.supermomentum("Bondi")
    assert rel(mine.mass_aspect(3).ndarray, -A._real_part(ref.data["psi2"][:, :16] + A.sf.modes_multiply(
        ref.data["sigma"], 2, 4, A.CubicSpline(ref.u, A.modes_bar(ref.data["sigma"], 2), axis=0).derivative()(ref.u), -2, 4, 3))) < RTOL


@pytest.mark.parametrize("n_times", [7000, 9000])
def test_transform_host_path_at_the_slab_thresholds(n_times):
    """The host path of WaveformGrid.transform switches strategy with size: below 8 MB the modes go up in one piece, from
    8 MB they stream in slabs, and from 8192 output times the tail is pipelined - the sizes around the switches against
    the oracle on a window, and against the device-resident path bit for bit."""
    t, data = smooth_modes(n_times=n_times, t0=0.0, t1=0.1 * n_times, seed=71)
    out = modes(t, data).transform(**BMS)
    plan = P.TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **BMS)
    u, m = plan.run(ops.to_device(t), ops.to_device(data))
    assert np.array_equal(out.t, u.cpu().numpy()) and np.array_equal(out.data, m.cpu().numpy())
    lo, hi = n_times // 2 - 300, n_times // 2 + 300
    ref = R.transform(R.Modes(t=t[lo:hi], data=data[lo:hi].copy()), **BMS)
    sel = np.searchsorted(out.t, ref.t[100:-100])
    assert np.array_equal(out.t[sel], ref.t[100:-100])
    assert rel(out.data[sel], ref.data[100:-100]) < 1e-10        # the window's own spline ends are ~1e-11 away after 100 steps


def test_transform_of_modes_in_page_locked_memory():
    """Modes that live in page-locked memory already (a numpy view of a pinned torch tensor): the library must neither try
    to register them (cudaHostRegister fails with "invalid argument" there, and the pending error used to surface at the
    next launch) nor release them; the result is the pageable-input result bit for bit, call after call."""
    import torch

    t, data = smooth_modes(n_times=30000, t0=0.0, t1=3000.0, seed=72)
    ref = modes(t, data).transform(**BMS)
    pinned = torch.empty(data.shape, dtype=torch.complex128, pin_memory=True)
    view = pinned.numpy()
    view[...] = data
    w = modes(t, data)
    w.data = view
    for _ in range(3):                      # second sighting is where pageable arrays get registered
        out = w.transform(**BMS)
        assert np.array_equal(out.t, ref.t) and np.array_equal(out.data, ref.data)
    lib = _lib.load()
    assert lib.scrib200_host_register(view.ctypes.data, view.nbytes) == 1      # "page-locked already", nothing to undo
    scratch = np.ones(1 << 20)
    assert lib.scrib200_host_register(scratch.ctypes.data, scratch.nbytes) == 0
    assert lib.scrib200_host_register(scratch.ctypes.data, scratch.nbytes) == 1
    assert lib.scrib200_host_unregister(scratch.ctypes.data) == 0


@pytest.mark.parametrize("bit_width", [8, 16, 32, 64])
def test_codec_stages_bit_exact(bit_width):
    """scri/utilities.py:194-407 on the GPU (scri_b200.utilities) against the oracle, bit for bit: multishuffle and its inverse
    for byte-wide, bit-wide and ragged piece widths and ragged lengths (the reference's tests/test_utilities.py:20-52, HDF5
    known answer included), the XOR transform of a mode series and its inverse, Fletcher-32 at lengths around the block size."""
    from oracle import utilities_ref as U
    from scri_b200 import utilities as ut

    dt = np.dtype(f"u{bit_width // 8}")
    rng = np.random.default_rng(123)
    for n in (1, 37, 5000):
        data = rng.integers(0, 2**bit_width, size=n, dtype=dt, endpoint=False)
        cases = [(1,) * bit_width, (8,) * (bit_width // 8), (bit_width,), tuple([3, 5] + [1] * (bit_width - 8))]
        if bit_width == 64:
            cases.append((8, 8, 4, 4, 4, 4) + (2,) * 8 + (1,) * 16)
        for widths in cases:
            sh = ut.multishuffle(widths)(data)
            assert sh.dtype == dt and np.array_equal(sh, U.multishuffle(widths)(data)), (n, widths)
            assert np.array_equal(ut.multishuffle(widths, forward=False)(sh), data), (n, widths)
        assert np.array_equal(ut.multishuffle((8,) * (bit_width // 8))(data), data.view(np.uint8).reshape(n, bit_width // 8).T.ravel().view(dt))
    with pytest.raises(ValueError):
        ut.multishuffle((8, 4))
    t, modes_ = smooth_modes(n_times=700 + bit_width, seed=81)
    x = modes_.copy()
    ref = U.xor_timeseries(modes_)
    out = ut.xor_timeseries(x)
    assert out is x and np.array_equal(x.view(np.uint64), ref.view(np.uint64))
    back = ut.xor_timeseries_reverse(x)
    assert np.array_equal(back.view(np.uint64), modes_.view(np.uint64))
    tt = t.copy()
    assert np.array_equal(ut.xor_timeseries(tt).view(np.uint64), U.xor_timeseries(t).view(np.uint64))     # 1-d series (w.t, corotating_paired_xor.py:88)
    for n in (2, 359, 360, 361, 100_003):
        d16 = rng.integers(0, 65536, size=n, dtype=np.uint16)
        assert ut.fletcher32(d16) == U.fletcher32(d16), n
    assert ut.fletcher32(modes_) == U.fletcher32(modes_)


# ------------------------------------------------------------------ round 2: full-size parity, frame branches, Nyquist
def test_config1_full_size_vs_oracle():
    """BASELINE configs[0] at its full size (fake_precessing_waveform, ell <= 8, 20 201 steps): to_corotating_frame against
    the oracle (oracle/frames_ref.py restates scri/mode_calculations.py:435-490 / scri/rotations.py:51-103 and is pinned
    by the reference's own output, tests/test_reference_golden.py) and the to_grid / from_grid round trip."""
    from oracle import frames_ref as FR

    w = sb.sample_waveforms.fake_precessing_waveform(t_1=2000.0)
    assert w.n_times == 20201
    ref = w.data.copy()
    Wo = R.Modes(t=w.t.copy(), data=ref.copy(), ell_min=2, ell_max=8)
    fo, omo = FR.corotating_frame(Wo, return_omega=True)
    wc, om = w.copy().to_corotating_frame(return_omega=True)
    assert rel(om, omo) < 1e-10
    # The frame solves dR/dt = omega R / 2 to `tolerance` = 1e-12 per step on both sides, by different Dormand-Prince
    # drivers; over 2000 M (several hundred orbits) the global errors reach 1e-7.  Both are therefore measured against
    # the same oracle integrated with a much tighter tolerance: the product must be at least as close to it as the
    # reference's algorithm is at the reference's tolerance, and the two must differ by no more than their own errors.
    f_tight = FR.corotating_frame(Wo, tolerance=1e-15)
    e_prod, e_orac = rel(wc.frame, f_tight), rel(fo, f_tight)
    print(f"corotating frame, 20201 steps: product vs tight {e_prod:.2e}, oracle(1e-12) vs tight {e_orac:.2e}, product vs oracle {rel(wc.frame, fo):.2e}")
    assert e_prod < max(1e-8, e_orac), (e_prod, e_orac)
    assert rel(wc.frame, fo) < 1e-8 + 2 * (e_prod + e_orac)
    Wr = R.rotate_decomposition_basis(Wo.copy(), wc.frame.copy())
    assert rel(wc.data, Wr.data) < RTOL                                  # same rotors: the rotation itself is exact to rounding
    assert rel(wc.copy().to_inertial_frame().data, ref) < RTOL
    g = w.to_grid()
    go = R.from_modes(R.Modes(t=w.t[::500].copy(), data=ref[::500].copy(), ell_min=2, ell_max=8))
    assert rel(g.data[::500], go.data) < RTOL
    back = sb.WaveformModes.from_grid(g, ell_max=8)
    assert rel(back.data, ref) < RTOL


def test_corotating_frame_reference_test_at_1e5_steps():
    """Port of the reference's tests/test_mode_calculations.py:112-126 at the size it asks for: a constant waveform turned
    by a known rotor series; corotating_frame must return that series to 1e-10 and to_corotating_frame the constant modes
    to 1e-8.  (In the reference `constant_waveform(end=10.0, n_times=100000)` only warns about the unknown keywords and
    runs on the default 1101 samples; here the 1e5 samples on [0, 10] are passed explicitly.)"""
    w = sb.sample_waveforms.constant_waveform(t=np.linspace(0.0, 10.0, 100000))
    omega = 2 * np.pi / 5.0
    R0 = quat.normalized(np.array([1.0, 2.0, 3.0, 4.0]))
    half = 0.5 * omega * w.t
    Rz = np.stack([np.cos(half), 0 * half, 0 * half, np.sin(half)], axis=-1)
    R_in = quat.mul(R0[None, :], Rz)
    w_rot = w.copy()
    w_rot.rotate_physical_system(R_in)
    R_out = sb.corotating_frame(w_rot, R0=R0, tolerance=1e-12)
    assert np.abs(R_in - R_out).max() < 1e-10, np.abs(R_in - R_out).max()
    w_rot.to_corotating_frame(R0=R0, tolerance=1e-12)
    assert np.abs(w_rot.data - w.data).max() < 1e-8 and w_rot.frameType == sb.Corotating
    Omega = quat.rotate_vector(R0, np.array([0.0, 0.0, omega]))
    w_rot2 = w.copy()
    w_rot2.rotate_physical_system(R_in)
    assert np.allclose(w_rot2.angular_velocity(), Omega[None, :], atol=1e-12, rtol=2e-8)   # :96-109


def test_frame_branches_vs_oracle():
    """Every branch of the frame functions that round 1 left unexecuted, against the oracle on the same input:
    corotating_frame(z_alignment_region=), to_corotating_frame(truncate_log_frame=True) in its two return shapes,
    angular_velocity(include_frame_velocity=True), to_coprecessing_frame(transition_times=), rotate_physical_system,
    minimal_rotation."""
    from oracle import frames_ref as FR, quat_series
    from scri_b200.mode_calculations import minimal_rotation

    w = sb.sample_waveforms.fake_precessing_waveform(t_0=-20.0, t_1=600.0, dt=0.25, ell_max=4)
    Wo = lambda: R.Modes(t=w.t.copy(), data=w.data.copy(), ell_min=2, ell_max=4)
    # rotor ODE: compared with the oracle's integrator at a far tighter tolerance (see test_config1_full_size_vs_oracle)
    fz = sb.corotating_frame(w.copy(), z_alignment_region=(0.1, 0.8))
    fz_tight = FR.corotating_frame(Wo(), z_alignment_region=(0.1, 0.8), tolerance=1e-15)
    assert rel(fz, fz_tight) < 1e-8, rel(fz, fz_tight)
    assert rel(fz, FR.corotating_frame(Wo(), z_alignment_region=(0.1, 0.8))) < 1e-6
    wt, om, lf = w.copy().to_corotating_frame(return_omega=True, truncate_log_frame=True, tolerance=1e-9)
    o, omo, lfo = FR.to_corotating_frame(Wo(), tolerance=1e-9, truncate_log_frame=True)
    q = 2.0 ** int(-np.floor(np.log2(2e-9)))
    assert lf.shape == lfo.shape and np.array_equal(lf * q, np.round(lf * q))       # on the lattice of the tolerance
    assert rel(wt.frame, quat.exp(lf)) < 1e-15                       # the frame IS exp(truncated log), to rounding
    assert rel(wt.frame, FR.corotating_frame(Wo(), tolerance=1e-15)) < 1e-6         # ODE at 1e-9 per step + one lattice step
    assert rel(wt.frame, quat.exp(lfo)) < 1e-5 and rel(om, omo) < 1e-10
    assert rel(wt.data, R.rotate_decomposition_basis(Wo(), wt.frame.copy()).data) < RTOL    # given the frame, the rotation is exact
    wc = w.copy().to_corotating_frame()
    # angular_velocity(include_frame_velocity=True) is checked against the reference's output in test_gpu_reference_golden.py
    wp = w.copy().to_coprecessing_frame(transition_times=(450.0, 520.0))
    op, fp = FR.to_coprecessing_frame(Wo(), transition_times=(450.0, 520.0))
    assert rel(wp.frame, fp) < 1e-7 and rel(wp.data, op.data) < 1e-7    # the damped tail is re-integrated: ODE tolerance again
    Rq = quat.normalized(np.array([0.3, -0.1, 0.7, 0.2]))
    a = w.copy()
    a.rotate_physical_system(Rq)
    b = R.rotate_decomposition_basis(Wo(), quat.conj(Rq))
    assert rel(a.data, b.data) < 1e-13
    assert rel(minimal_rotation(wc.frame, w.t, 3), quat_series.minimal_rotation(wc.frame, w.t, 3)) < 1e-12


def test_config5_full_size_fluxes_and_dominant_eigenvector():
    """BASELINE configs[4] at its full size (1e6 steps, ell <= 16): energy / momentum / angular-momentum flux and
    LLDominantEigenvector against the oracle on windows (interior rows: the window's own spline ends differ), plus the
    size-independent properties: quadratic scaling, E >= 0, unit and sign-continuous eigenvector."""
    N = 1_000_000
    t, data = smooth_modes(n_times=N, ell_max=16, t0=0.0, t1=1e5, seed=31)
    w = modes(t, data, ell_max=16)
    E, p, J = w.energy_flux(), w.momentum_flux(), w.angular_momentum_flux()
    dpa = w.LLDominantEigenvector()
    assert E.shape == (N,) and p.shape == (N, 3) and J.shape == (N, 3) and dpa.shape == (N, 3)
    assert (E >= 0).all()
    assert np.abs(np.sum(dpa * dpa, axis=1) - 1).max() < 1e-13
    # (no global sign property: the reference flips a step only when it is more than 60 degrees from its neighbour,
    # mode_calculations.py:380-399, and random modes do cross eigenvalues; the windows below check the signs it produces)
    for lo in (0, 499_000, N - 1200):
        hi = lo + 1200
        Wo = R.Modes(t=t[lo:hi], data=data[lo:hi].copy(), ell_min=2, ell_max=16)
        a, b = (0 if lo == 0 else 200), (1200 if hi == N else 1000)      # keep the true series ends, drop the window's own
        assert rel(E[lo + a : lo + b], R.energy_flux(Wo)[a:b]) < 1e-11
        assert rel(p[lo + a : lo + b], R.momentum_flux(Wo)[a:b]) < 1e-11
        assert rel(J[lo + a : lo + b], R.angular_momentum_flux(Wo)[a:b]) < 1e-11
        do = R.LLDominantEigenvector(Wo, RoughDirection=dpa[lo], RoughDirectionIndex=0)
        assert rel(dpa[lo:hi], do) < 1e-11
    w2 = modes(t[:200_000], 3.0 * data[:200_000], ell_max=16)
    assert np.allclose(w2.energy_flux()[:-100], 9 * E[:199_900], rtol=1e-11)


def test_theta_nyquist_content_of_the_remapped_grid():
    """spinsfast.map2salm on input that is not band limited is the one behaviour of the third-party code the oracle can
    only follow from the published algorithm: the ring's Nyquist frequency p = N_theta - 1 enters the theta weights once
    (oracle/spinsfast.py, scri_b200/_sf.py) - an implementation could also count it twice or drop it.  For band-limited
    input the readings coincide exactly.  This test MEASURES what the choice is worth on the grid the headline config
    (configs[1]: ell <= 8 on 25 x 25, supertranslation + rotation + boost 0.037) feeds the analysis: while the boost has
    moved the retarded times of the grid points apart by less than a wave period (|u'| of a few hundred M) the three readings
    agree to ~1e-9 of the modes or better; by u' ~ 9000 M the time shift across the sphere is +-330 M, i.e. +-100 rad of
    wave phase on a grid whose Nyquist frequency is 12: the field is thoroughly aliased, the transformed modes are no longer
    meaningful in ANY implementation, and the readings differ at the 1e-3 level.  DESIGN.md section 2 states this as the one
    parity item that cannot be pinned without running spinsfast itself."""
    from scri_b200 import _sf

    w = sb.sample_waveforms.fake_precessing_waveform(t_0=-20.0, t_1=9400.0, dt=0.1)
    plan = P.TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **BMS)
    u, grid = plan.run(ops.to_device(w.t), ops.to_device(w.data), return_grid=True)
    n_theta, n_phi, L = plan.n_theta, plan.n_phi, 8
    assert (n_theta, n_phi) == (25, 25)
    E, Wt = _sf.analysis_tables(-2, 2, L, n_theta, n_phi)
    Nn = n_theta - 1
    theta = np.pi * np.arange(n_theta) / Nn
    dq = 2.0 * (2.0 / (1.0 - Nn * Nn) * np.cos(Nn * theta)) / (2 * Nn)     # the p = N term's share of q_j
    dq[0] *= 0.5
    dq[-1] *= 0.5
    q = _sf.clenshaw_curtis_theta_weights(n_theta)
    ms = np.concatenate([np.arange(-l, l + 1) for l in range(2, L + 1)]) + L
    worth = {}
    for name, rows in (("early", slice(0, 3000, 7)), ("late", slice(-4000, None, 7))):
        gr = grid[rows].cpu().numpy().reshape(-1, n_theta, n_phi)
        fm = np.einsum("tjk,km->tjm", gr, E)                                # phi-DFT
        once = np.einsum("nj,tjn->tn", Wt, fm[:, :, ms])
        delta = np.einsum("nj,tjn->tn", Wt * (dq / q)[None, :], fm[:, :, ms])   # counting the term once more / once less
        assert rel(plan.analyze(torch_from(gr.reshape(gr.shape[0], -1))).cpu().numpy(), once) < 1e-13
        worth[name] = float(np.abs(delta).max() / np.abs(once).max())
    print(f"theta-Nyquist term, relative to the modes: early {worth['early']:.2e}, late {worth['late']:.2e}")
    assert worth["early"] < 1e-8 and worth["late"] < 1e-2, worth


def torch_from(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def test_empty_retained_block():
    """A window so late that, under the boost, no output time lies inside the span covered by every grid point
    (waveform_grid.py:564-568 keeps nothing): the reference returns a waveform without time steps; so does the product."""
    w = sb.sample_waveforms.fake_precessing_waveform(t_0=8980.0, t_1=9400.0, dt=0.1)
    ref = R.transform(R.Modes(t=w.t.copy(), data=w.data.copy()), **BMS)
    assert ref.t.shape[0] == 0
    out = w.transform(**BMS)
    assert out.t.shape == (0,) and out.data.shape == (0, 77) and out.ell_max == 8


def test_abd_conformal_factors_reference_test():
    """Port of the reference's tests/test_asymptoticbondidata.py:33-93 (ell_max = 32, tolerance 4e-14): the conformal factors
    k, eth(k)/k, 1/k, 1/k^3 on the boosted grid (scri/asymptotic_bondi_data/transformations.py:150-196) against their
    evaluation from modes - 1/k and k analysed on the undistorted 65 x 65 grid (map2salm on the GPU), resynthesized on the
    distorted rotors."""
    from scri_b200 import _sf
    from scri_b200.asymptotic_bondi_data import boosted_grid, conformal_factors

    tolerance = 4e-14
    ell_max = 32
    n_theta = n_phi = 2 * ell_max + 1
    v = np.array([0.01, 0.02, 0.03])
    gamma = 1 / np.sqrt(1 - v @ v)
    Rg = boosted_grid(np.array([1.0, 0.0, 0.0, 0.0]), v, n_theta, n_phi)
    k, ethk_over_k, one_over_k, one_over_k3 = conformal_factors(v, Rg)
    assert k.shape == ethk_over_k.shape == one_over_k.shape == one_over_k3.shape == (1, n_theta, n_phi)
    theta = np.linspace(0.0, np.pi, n_theta)[:, None]
    phi = np.linspace(0.0, 2 * np.pi, n_phi, endpoint=False)[None, :]
    kinv = gamma * (1 - v[0] * np.sin(theta) * np.cos(phi) - v[1] * np.sin(theta) * np.sin(phi) - v[2] * np.cos(theta))
    kappa_inv = ops.map2salm(kinv[None].astype(complex), 0, ell_max, n_theta, n_phi)[0]
    kappa = ops.map2salm((1 / kinv)[None].astype(complex), 0, ell_max, n_theta, n_phi)[0]
    Y0 = _sf.SWSH_grid(Rg.reshape(-1, 4), 0, ell_max)
    one_over_k2 = (Y0 @ kappa_inv).reshape(n_theta, n_phi)
    ell = np.concatenate([np.full(2 * l + 1, l) for l in range(ell_max + 1)]).astype(float)
    eth_kappa = kappa * np.sqrt(ell * (ell + 1) / 2.0)                       # sf.eth_GHP on spin 0
    ethk2 = (_sf.SWSH_grid(Rg.reshape(-1, 4), 1, ell_max) @ eth_kappa).reshape(n_theta, n_phi)
    k2 = 1 / one_over_k2
    errs = [float(np.abs(a - b).max()) for a, b in ((k[0], k2), (ethk_over_k[0], ethk2 / k2), (one_over_k[0], one_over_k2), (one_over_k3[0], one_over_k2**3))]
    print("conformal factors vs their mode expansion (max abs difference):", errs)
    # The reference asserts 4e-14 for all four.  The check path here (and in the oracle: oracle.spinsfast gives the same
    # figures) carries a rounding floor of 1.5e-15 on every one of the 1089 modes of k (|k_00| = 3.5); eth multiplies
    # the ell = 32 floor by 23 before 1089 of them are summed on the grid, which is the 3e-13 seen on eth(k)/k.  The
    # functions under test agree with the reference's own output to 1e-14 (test_gpu_reference_golden.py).
    assert errs[0] < tolerance and errs[2] < tolerance and errs[3] < 1e-13 and errs[1] < 1e-12, errs


def test_captured_transform_replays_the_eager_path():
    """TransformPlan.capture: the device-resident step recorded as one CUDA graph gives the eager path's result bit for bit,
    follows new contents of its input tensors, and its baked-in retained block is verified after the replay."""
    import torch

    t, data = smooth_modes(n_times=20000, t0=0.0, t1=2000.0, seed=91)
    plan = P.TransformPlan(2, 8, sb.h, r_is_scaled_out=True, **BMS)
    td, ad = ops.to_device(t), ops.to_device(data)
    u1, m1 = plan.run(td, ad)
    cap = plan.capture(td, ad)
    u2, m2 = cap.replay()
    assert cap.verify()
    assert torch.equal(u1, u2) and torch.equal(m1, m2)
    ad.mul_(2.0)                                   # same tensor, new contents: h is linear in the modes up to the supertranslation term
    u3, m3 = cap.replay()
    torch.cuda.synchronize()
    u4, m4 = plan.run(td, ad)
    assert torch.equal(u3, u4) and torch.equal(m3, m4)
