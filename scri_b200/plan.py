"""Host-side planning for the BMS transformation and the device pipeline that executes it.

`process_transformation_kwargs` mirrors scri/waveform_grid.py:20-190 (same keyword names, defaults,
validation and exception types); it is O(G) host work done once per call, exactly as in the
reference.  `TransformPlan` turns its result into device-resident tables and runs the three
kernels of the path (SWSH synthesis -> retarded-time spline remap -> SWSH analysis) through the
C ABI in include/scrib200.h.
"""
import math
import pprint
import warnings

import numpy as np

from . import _lib, _sf
from . import _quaternion as Q
from .constants import ConformalWeights, DataNames, RScaling, SpinWeights, h, hdot, news, psi0, psi1, psi2, psi3, psi4, sigma


def boosted_rotor_grid(frame_rotation, boost_velocity, n_theta, n_phi):
    """Rotors of the output (theta', phi') grid carried back to the input frame, R = B'(theta, phi) R_frame R_{theta'phi'}
    (scri/waveform_grid.py:130-174 and scri/asymptotic_bondi_data/transformations.py:100-148), vectorised.
    Returns (R_j_k [n_theta, n_phi, 4], thetaprm_phiprm [n_theta, n_phi, 2])."""
    beta = np.linalg.norm(boost_velocity)
    varphi = math.atanh(beta)
    thetaprm = np.linspace(0.0, np.pi, num=n_theta, endpoint=True)
    phiprm = np.linspace(0.0, 2 * np.pi, num=n_phi, endpoint=False)
    thetaprm_j_phiprm_k = np.stack(np.meshgrid(thetaprm, phiprm, indexing="ij"), axis=-1)
    rotated = Q.qmul(frame_rotation, Q.from_spherical_coords(thetaprm_j_phiprm_k[..., 0], thetaprm_j_phiprm_k[..., 1]))
    if beta > 3e-14:
        vhat = boost_velocity / beta
        th, ph = Q.as_spherical_coords(rotated)
        rprm = np.stack([np.cos(ph) * np.sin(th), np.sin(ph) * np.sin(th), np.cos(th)], axis=-1)
        Thetaprm = np.arccos(np.clip(rprm @ vhat, -1.0, 1.0))
        Theta = 2 * np.arctan(math.exp(-varphi) * np.tan(Thetaprm / 2.0))
        cross = np.cross(rprm, vhat)
        cn = np.sqrt(np.sum(cross * cross, axis=-1))
        safe = cn > 1e-200
        nhat = np.where(safe[..., None], cross / np.where(safe, cn, 1.0)[..., None], 0.0)
        B = Q.qexp_vec(nhat * ((Thetaprm - Theta) / 2)[..., None])
        B[~safe] = np.array([1.0, 0.0, 0.0, 0.0])
        R_j_k = Q.qmul(B, rotated)
    else:
        R_j_k = rotated
    return R_j_k, thetaprm_j_phiprm_k


def process_transformation_kwargs(ell_max, **kwargs):
    """Parse the BMS-transformation keywords (scri/waveform_grid.py:20-190).

    Returns (supertranslation, ell_max_supertranslation, ell_max, n_theta, n_phi, boost_velocity, beta,
    gamma, varphi, R_j_k, thetaprm_phiprm, kwargs) - `R_j_k` is a float array [n_theta, n_phi, 4].
    """
    supertranslation = np.zeros((4,), dtype=complex)
    ell_max_supertranslation = 1
    if "supertranslation" in kwargs:
        supertranslation = np.array(kwargs.pop("supertranslation"), dtype=complex)
        if supertranslation.dtype != "complex" and supertranslation.size > 0:
            raise TypeError(
                "\nInput argument `supertranslation` should be a complex array with size>0.\n"
                f"Got a {supertranslation.dtype} array of shape {supertranslation.shape}."
            )
        if supertranslation.size <= 4:
            supertranslation = np.pad(supertranslation, (0, 4 - supertranslation.size), "constant", constant_values=(0.0,))
        ell_max_supertranslation = int(np.sqrt(len(supertranslation))) - 1
        if (ell_max_supertranslation + 1) ** 2 != len(supertranslation):
            raise ValueError(
                "\nInput supertranslation parameter must contain modes from ell=0 up to some ell_max, including\n"
                "all relevant m modes in standard order.  Thus, it must be an array with length given by a "
                f"perfect square; its length is {len(supertranslation)}"
            )
        for ell in range(ell_max_supertranslation + 1):
            for m in range(ell + 1):
                i_pos = _sf.LM_index(ell, m, 0)
                i_neg = _sf.LM_index(ell, -m, 0)
                a = supertranslation[i_pos]
                b = supertranslation[i_neg]
                if abs(a - (-1.0) ** m * b.conjugate()) > 3e-16 + 1e-15 * abs(b):
                    raise ValueError(
                        f"\nsupertranslation[{i_pos}]={a}  # (ell,m)=({ell},{m})\n"
                        f"supertranslation[{i_neg}]={b}  # (ell,m)=({ell},{-m})\n"
                        "Will result in an imaginary supertranslation."
                    )
    s4pi = math.sqrt(4 * math.pi)
    c1 = math.sqrt(2 * math.pi / 3)
    c0 = math.sqrt(4 * math.pi / 3)

    def vector_as_ell_1_modes(v):
        return np.array([c1 * (v[0] + 1j * v[1]), c0 * v[2], c1 * (-v[0] + 1j * v[1])], dtype=complex)

    def vector_from_ell_1_modes(a):
        return np.array([(a[0] - a[2]) / (2 * c1), (a[0] + a[2]) / (2j * c1), a[1] / c0])

    spacetime_translation = np.zeros((4,), dtype=float)
    spacetime_translation[0] = (supertranslation[0] / s4pi).real
    spacetime_translation[1:4] = -vector_from_ell_1_modes(supertranslation[1:4]).real
    if "spacetime_translation" in kwargs:
        st_trans = np.array(kwargs.pop("spacetime_translation"), dtype=float)
        if st_trans.shape != (4,) or st_trans.dtype != "float":
            raise TypeError(
                "\nInput argument `spacetime_translation` should be a float array of shape (4,).\n"
                f"Got a {st_trans.dtype} array of shape {st_trans.shape}."
            )
        spacetime_translation = st_trans[:]
        supertranslation[0] = spacetime_translation[0] * s4pi
        supertranslation[1:4] = vector_as_ell_1_modes(-spacetime_translation[1:4])
    if "space_translation" in kwargs:
        s_trans = np.array(kwargs.pop("space_translation"), dtype=float)
        if s_trans.shape != (3,) or s_trans.dtype != "float":
            raise TypeError(
                "\nInput argument `space_translation` should be an array of floats of shape (3,).\n"
                f"Got a {s_trans.dtype} array of shape {s_trans.shape}."
            )
        spacetime_translation[1:4] = s_trans[:]
        supertranslation[1:4] = vector_as_ell_1_modes(-spacetime_translation[1:4])
    if "time_translation" in kwargs:
        t_trans = kwargs.pop("time_translation")
        if not isinstance(t_trans, float):
            raise TypeError(f"\nInput argument `time_translation` should be a single float.\nGot {t_trans}.")
        spacetime_translation[0] = t_trans
        supertranslation[0] = spacetime_translation[0] * s4pi

    w_ell_max = ell_max
    ell_max = w_ell_max + ell_max_supertranslation
    n_theta = kwargs.pop("n_theta", 2 * ell_max + 1)
    n_phi = kwargs.pop("n_phi", 2 * ell_max + 1)
    if n_theta < 2 * ell_max + 1 and abs(supertranslation[1:]).max() > 0.0:
        warnings.warn(
            f"n_theta={n_theta} is small; because of the supertranslation, "
            f"it will lose accuracy for anything less than 2*ell+1={ell_max}"
        )
    if n_theta < 2 * w_ell_max + 1:
        raise ValueError(f"n_theta={n_theta} is too small; must be at least 2*ell+1={2 * w_ell_max + 1}")
    if n_phi < 2 * ell_max + 1 and abs(supertranslation[1:]).max() > 0.0:
        warnings.warn(
            f"n_phi={n_phi} is small; because of the supertranslation, "
            f"it will lose accuracy for anything less than 2*ell+1={ell_max}"
        )
    if n_phi < 2 * w_ell_max + 1:
        raise ValueError(f"n_phi={n_phi} is too small; must be at least 2*ell+1={2 * w_ell_max + 1}")

    frame_rotation = Q.as_float_quat(np.array(kwargs.pop("frame_rotation", [1, 0, 0, 0]), dtype=float))
    if Q.qabs(frame_rotation) < 3e-16:
        raise ValueError(f"frame_rotation={frame_rotation} should be a unit quaternion")
    frame_rotation = Q.qnormalized(frame_rotation)

    boost_velocity = np.array(kwargs.pop("boost_velocity", [0.0] * 3), dtype=float)
    beta = np.linalg.norm(boost_velocity)
    if boost_velocity.shape != (3,) or beta >= 1.0:
        raise ValueError(
            f"Input boost_velocity=`{boost_velocity}` should be a 3-vector with magnitude strictly less than 1.0."
        )
    gamma = 1 / math.sqrt(1 - beta**2)
    varphi = math.atanh(beta)

    R_j_k, thetaprm_j_phiprm_k = boosted_rotor_grid(frame_rotation, boost_velocity, n_theta, n_phi)

    return (
        supertranslation,
        ell_max_supertranslation,
        ell_max,
        n_theta,
        n_phi,
        boost_velocity,
        beta,
        gamma,
        varphi,
        R_j_k,
        thetaprm_j_phiprm_k,
        kwargs,
    )


def _ell_factors(n, fn):
    out = np.zeros(n)
    i = 0
    ell = 0
    while i < n:
        for m in range(-ell, ell + 1):
            out[i] = fn(ell)
            i += 1
        ell += 1
    return out


def pack_synthesis_matrix(Y, ell_min, ell_max):
    """Real GEMM operand for scrib200_swsh_synthesize from Y[g, LM_index(l,m,0)] (complex).

    B[2lm, 2g] = Re Y, B[2lm+1, 2g] = -Im Y, B[2lm, 2g+1] = Im Y, B[2lm+1, 2g+1] = Re Y, zero padded to
    [roundup(2n,16), roundup(2G,64)].
    """
    G = Y.shape[0]
    Ys = Y[:, ell_min * ell_min : (ell_max + 1) ** 2]
    n = Ys.shape[1]
    Kpad = -(-2 * n // 16) * 16
    Ncpad = -(-2 * G // 64) * 64
    B = np.zeros((Kpad, Ncpad))
    B[0 : 2 * n : 2, 0 : 2 * G : 2] = Ys.real.T
    B[1 : 2 * n : 2, 0 : 2 * G : 2] = -Ys.imag.T
    B[0 : 2 * n : 2, 1 : 2 * G : 2] = Ys.imag.T
    B[1 : 2 * n : 2, 1 : 2 * G : 2] = Ys.real.T
    return B, Kpad, Ncpad


_blas_controller = None


def _quiet_blas():
    """The plan's host algebra is a handful of tiny matrix products; run them on one BLAS thread.  A multi-threaded
    BLAS leaves its 16 workers spinning for tens of milliseconds after each call, which is exactly when the pinned
    staging copy of the waveform wants the cores (measured: 3 ms -> 10 ms for 124 MB)."""
    global _blas_controller
    try:
        if _blas_controller is None:
            from threadpoolctl import ThreadpoolController

            _blas_controller = ThreadpoolController()   # introspecting the loaded libraries costs ~2 ms: do it once
        return _blas_controller.limit(limits=1, user_api="blas")
    except Exception:  # threadpoolctl missing: correctness does not depend on it
        import contextlib

        return contextlib.nullcontext()


class GridPlan:
    """What every transformation shares once the rotor grid is fixed: the conformal factor and supertranslation on the
    grid (device arrays `d_k`, `d_alpha`), the output time axis, and the synthesis, spline remap and analysis launches.
    `divide_by_gamma`: u' = (t - dt) / gamma as the ABD path forms it (transformations.py:393); otherwise
    u' = (1/gamma)(t - dt) as in waveform_grid.py:565."""

    def __init__(self, device, n_theta, n_phi, gamma, time_translation, kconformal, alpha, divide_by_gamma=False):
        torch = _lib.require_cuda()
        _lib.load()
        self.torch = torch
        self.device = torch.device(device)
        self.n_theta, self.n_phi = int(n_theta), int(n_phi)
        self.G = self.n_theta * self.n_phi
        self.gamma = gamma
        self.time_translation = time_translation
        self.divide_by_gamma = divide_by_gamma
        self.kconformal, self.alpha = kconformal, alpha
        self.d_k = torch.from_numpy(np.ascontiguousarray(kconformal)).to(self.device)
        self.d_alpha = torch.from_numpy(np.ascontiguousarray(alpha)).to(self.device)
        self._ws = None
        self._d2h_stream = None
        self._side = None
        self._host_pool = []
        self.spline_halo = 0   # 0 = chosen from the decay diagnostics of scrib200_spline_prepare
        self.spline_body = 0   # 0 = default intervals per tile

    def _side_stream(self):
        if self._side is None:
            self._side = self.torch.cuda.Stream(device=self.device)
        return self._side

    def _info_host(self):
        """A pinned 64-byte landing buffer for `info` (recycled: no allocation in steady state)."""
        if self._host_pool:
            return self._host_pool.pop()
        return self.torch.empty(8, dtype=self.torch.float64, pin_memory=True)

    def prepare(self, t, overlapped=False, after=None, speculate=False, memo_key=None):
        """Launch the per-time-axis preparation (scrib200_spline_prepare): spline factor table, u' for every sample,
        the retained block and the decay diagnostics.  Nothing is read back here; see `TimePrep.resolve`.
        `overlapped=True` launches on the plan's side stream so the (tiny, latency-bound) kernels run under the
        synthesis GEMM; the caller's stream must then `wait_event(prep.done)` before it consumes the tables.  `after`
        (an event recorded when `t` became ready) lets the side stream start without waiting for work queued since.
        `speculate=True`: if this very tensor (same storage, same version counter, same length) was prepared before, the
        retained block and halo found then are assumed at once, so the caller can queue every later launch without waiting
        for the 64-byte read-back in the middle of the step; `TimePrep.verify()` compares with what the kernels found
        this time (and the caller repeats the step in the rare case they differ)."""
        prep = TimePrep(self, t, overlapped, after)
        if speculate:
            if not hasattr(self, "_prep_memo"):
                self._prep_memo = {}
            prep._memo = self._prep_memo
            # identity of the time axis: the device tensor itself, or what the caller says (a host array that is uploaded
            # afresh on every call); a stale identity costs one repeated step, never a wrong result (see verify)
            prep._memo_key = memo_key if memo_key is not None else (t.data_ptr(), getattr(t, "_version", 0), int(t.shape[0]))
            seen = self._prep_memo.get(prep._memo_key)
            if seen is not None:
                prep._assumed = seen
        return prep

    def output_times(self, t, t_ends=None):
        """u'_i and the retained block (waveform_grid.py:564-568) as a device tensor.  `t_ends` is accepted for
        backward compatibility and ignored (the block is found on the device)."""
        return self.prepare(t).uprm

    def _remap(self, t, F, uprm, prep, tile, n_series=1, rows_needed=None, out=None):
        """F [n_series * N, G] (series stacked along time) -> remapped grid; rows b*n_out.. belong to series b.
        `rows_needed` = (row_lo, row_hi): the caller knows that these output times read input rows [row_lo, row_hi) only
        (`input_rows_for_outputs`); only the tiles holding them are launched."""
        torch = self.torch
        lib = _lib.load()
        if prep is None:
            prep = self.prepare(t)
        N, n_out = t.shape[0], uprm.shape[0]
        rows = n_out * n_series
        if out is not None:
            pass                                   # caller's buffer (scratch of the streaming pipeline)
        elif tile:
            out = torch.empty((-(-rows // tile), self.G, tile), dtype=torch.complex128, device=self.device)
        else:
            out = torch.empty((rows, self.G), dtype=torch.complex128, device=self.device)
        if rows == 0:          # no output time inside the span every grid point covers: an empty result, as in the reference
            return out
        halo, body = prep.halo_body(self.spline_halo, self.spline_body)
        need = lib.scrib200_spline_remap_workspace_bytes(N, self.G, halo, body)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        if rows_needed is not None:
            _lib.check(
                lib.scrib200_spline_remap_rows(
                    _lib.ptr(t), N, _lib.ptr(F), self.G, _lib.ptr(self.d_k), _lib.ptr(self.d_alpha), _lib.ptr(prep.tab),
                    _lib.ptr(uprm), n_out, _lib.ptr(out), tile, halo, body, n_series, int(rows_needed[0]), int(rows_needed[1]),
                    _lib.ptr(self._ws), self._ws.numel(), _lib.stream_ptr(),
                ),
                "spline_remap_rows",
            )
            return out
        _lib.check(
            lib.scrib200_spline_remap(
                _lib.ptr(t), N, _lib.ptr(F), self.G, _lib.ptr(self.d_k), _lib.ptr(self.d_alpha), _lib.ptr(prep.tab),
                _lib.ptr(uprm), n_out, _lib.ptr(out), tile, halo, body, n_series, _lib.ptr(self._ws), self._ws.numel(),
                _lib.stream_ptr(),
            ),
            "spline_remap",
        )
        return out

    def input_rows_for_outputs(self, t_host, u_first, u_last):
        """[row_lo, row_hi): the input samples any grid point can need for output times in [u_first, u_last].  Grid point g
        evaluates its spline at x = u, x_i = k_g (t_i - alpha_g), i.e. inside the input interval around t = u / k_g +
        alpha_g: the extremes over the grid, widened by two samples."""
        k = np.asarray(self.kconformal, dtype=float).ravel()
        al = np.asarray(self.alpha, dtype=float).ravel()
        t_lo = float(np.min(u_first / k + al))
        t_hi = float(np.max(u_last / k + al))
        lo = int(np.searchsorted(t_host, t_lo, side="left")) - 3
        hi = int(np.searchsorted(t_host, t_hi, side="right")) + 3
        return max(lo, 0), min(hi, int(t_host.shape[0]))

    def remap(self, t, F, uprm, prep=None):
        """Spline each grid point's series from knots k(t-alpha) onto u' (waveform_grid.py:576-588); [N', G]."""
        return self._remap(t, F, uprm, prep, 0)

    def synthesize_with(self, data, d_B, n_modes, Kpad, Ncpad, d_offset, d_scale, out=None, d_B3=None, folded=False):
        """Synthesis of `data` [rows, n_modes] complex128 against the packed table `d_B` (pack_synthesis_matrix layout), one
        launch into `out` [rows, G] (allocated when None).  By default the three-multiplication kernel on the table's three
        real planes Y_r, Y_i, Y_r + Y_i: `d_B3` when the caller keeps them, else packed here (one pass over the table,
        ~0.3 ms at ell_max = 32) and freed after, so that fields synthesized one after the other never hold two sets.  On the
        FP64 tensor pipe (92 % DMMA activity in round 1) 6 n G flops instead of 8 n G is a quarter of the time.  `folded`,
        or SCRIB200_SYNTH_FOLDED set, takes the one-GEMM form instead; the two round differently, so each caller keeps
        the kernel it has."""
        import os

        torch = self.torch
        lib = _lib.load()
        rows = data.shape[0]
        if out is None:
            out = torch.empty((rows, self.G), dtype=torch.complex128, device=self.device)
        if folded or os.environ.get("SCRIB200_SYNTH_FOLDED"):
            _lib.check(
                lib.scrib200_swsh_synthesize(
                    _lib.ptr(data), rows, n_modes, _lib.ptr(d_B), Kpad, Ncpad, _lib.ptr(d_offset), _lib.ptr(d_scale), self.G,
                    _lib.ptr(out), _lib.stream_ptr(),
                ),
                "swsh_synthesize",
            )
            return out
        npad3, Gpad3 = -(-n_modes // 8) * 8, -(-self.G // 32) * 32
        if d_B3 is None:
            d_B3 = torch.empty((3, npad3, Gpad3), dtype=torch.float64, device=self.device)
            _lib.check(lib.scrib200_swsh_pack3m(_lib.ptr(d_B), Kpad, Ncpad, n_modes, self.G, _lib.ptr(d_B3), npad3, Gpad3, _lib.stream_ptr()),
                       "swsh_pack3m")
        _lib.check(
            lib.scrib200_swsh_synthesize_3m(_lib.ptr(data), rows, n_modes, _lib.ptr(d_B3), npad3, Gpad3, _lib.ptr(d_offset), _lib.ptr(d_scale),
                                            self.G, _lib.ptr(out), _lib.stream_ptr()),
            "swsh_synthesize_3m",
        )
        return out

    def analyze(self, grid, analysis=None):
        """[N', G] complex128, time-major -> [N', n_modes_out] (waveform_grid.py:303-307) by `analysis` (ops.analysis;
        default the plan's own): large band limits take the separable tensor-core analysis, the rest the shared-memory
        kernels (ops.analyze)."""
        from . import ops

        an = analysis or self.analysis
        if grid.shape[0] == 0:
            return self.torch.empty((0, an.n_modes), dtype=self.torch.complex128, device=self.device)
        return ops.analyze(grid, an)

    def analyze_tiled(self, gridT, n_out, out=None, analysis=None):
        """gridT [ceil(n_out/T), G, T] complex128 (time-tiled, T = the analysis' tile) -> [n_out, n_modes_out]."""
        an = analysis or self.analysis
        torch = self.torch
        if out is None:
            out = torch.empty((n_out, an.n_modes), dtype=torch.complex128, device=self.device)
        if n_out == 0:
            return out
        _lib.check(
            _lib.load().scrib200_map2salm_tiled(
                _lib.ptr(gridT), an.tile, n_out, self.n_theta, self.n_phi, _lib.ptr(an.trig), _lib.ptr(an.Wt), an.ell_min, an.ell_max,
                _lib.ptr(out), _lib.stream_ptr(),
            ),
            "map2salm_tiled",
        )
        return out

    def remap_analyze(self, t, F, uprm, prep, analysis, n_series=1, rows_needed=None, grid_out=None, out=None):
        """Spline remap of F [n_series * N, G] onto u' and the analysis `analysis` (ops.analysis) of the result:
        [n_series * N', n_modes].  The remapped grid is handed over time-tiled (scrib200_spline_remap with the analysis'
        tile, then scrib200_map2salm_tiled) when the analysis has a tile, time-major (`remap`, `analyze`) when its tables
        are too large for that.  `rows_needed` as for `_remap`; `grid_out` and `out` are caller buffers for the tiled
        grid and the modes of the tiled path."""
        n_out = n_series * uprm.shape[0]
        grid = self._remap(t, F, uprm, prep, analysis.tile, n_series, rows_needed, grid_out)
        if analysis.tile:
            return self.analyze_tiled(grid, n_out, out, analysis)
        return self.analyze(grid, analysis)

    def weyl_mix(self, fields, coefs, t, d_A, d_C, d_scale, d_offset, out):
        """One scrib200_weyl_mix launch (see include/scrib200.h)."""
        import ctypes

        ptrs = (ctypes.c_void_p * len(fields))(*[f.data_ptr() for f in fields])
        cf = (ctypes.c_double * len(coefs))(*[float(c) for c in coefs])
        _lib.check(
            _lib.load().scrib200_weyl_mix(
                ptrs, cf, len(fields), _lib.ptr(t), t.shape[0], self.G, _lib.ptr(self.d_alpha), _lib.ptr(d_A), _lib.ptr(d_C),
                _lib.ptr(d_scale), _lib.ptr(d_offset) if d_offset is not None else None, _lib.ptr(out), _lib.stream_ptr(),
            ),
            "weyl_mix",
        )
        return out


class TransformPlan(GridPlan):
    """Device-resident tables for one BMS transformation of one kind of waveform.

    Built from the same quantities scri/waveform_grid.py:431-474 computes on the host (rotor grid,
    SWSH tables, conformal factor, supertranslation on the grid); executed by `run`.
    """

    def __init__(self, ell_min, ell_max, dataType, r_is_scaled_out=True, out_ell_max=None, device="cuda", **kwargs):
        with _quiet_blas():
            self._build(ell_min, ell_max, dataType, r_is_scaled_out, out_ell_max, device, kwargs)

    def _build(self, ell_min, ell_max, dataType, r_is_scaled_out, out_ell_max, device, kwargs):
        self.ell_min, self.ell_max, self.dataType = int(ell_min), int(ell_max), int(dataType)
        self.spin_weight = SpinWeights[self.dataType]
        self.conformal_weight = ConformalWeights[self.dataType] - (RScaling[self.dataType] if r_is_scaled_out else 0)
        (
            supertranslation,
            ell_max_st,
            L,
            n_theta,
            n_phi,
            boost_velocity,
            beta,
            gamma,
            varphi,
            R_j_k,
            _,
            leftover,
        ) = process_transformation_kwargs(self.ell_max, **kwargs)
        self.leftover_kwargs = leftover
        self.supertranslation = supertranslation
        self.L, self.beta = L, beta
        self.out_ell_max = self.ell_max if out_ell_max is None else int(out_ell_max)
        self.out_ell_min = abs(self.spin_weight)
        s = self.spin_weight

        R = R_j_k.reshape(-1, 4)
        # the big table sY_lm(R_g) for the waveform's own modes is built on the device (scrib200_swsh_pack); the host only
        # needs the few columns l <= ell_max_st that enter the constant corrections below
        Y = _sf.SWSH_grid(R, s, ell_max_st) if self.dataType in (h, sigma) else None
        SH = _sf.SWSH_grid(R, 0, ell_max_st)
        rhat = Q.rotate_z(R)
        kconformal = 1.0 / (gamma * (1 - rhat @ boost_velocity))
        super().__init__(device, n_theta, n_phi, gamma, (supertranslation[0] / math.sqrt(4 * math.pi)).real, kconformal,
                         (SH @ supertranslation).real)
        torch = self.torch
        offset_c = np.zeros(self.G, dtype=complex)
        self.mix = []          # higher Weyl scalars mixed into psi0..psi3 (empty for every other data type)
        nontrivial = beta != 0 or (supertranslation[1:] != 0).any()
        if nontrivial:
            nst = (ell_max_st + 1) ** 2
            if self.dataType == h:
                # 2 ethbar ethbar alpha (GHP): factor sqrt((l-1) l (l+1) (l+2))   (waveform_grid.py:486-494)
                fac = _ell_factors(nst, lambda l: math.sqrt(max((l - 1) * l * (l + 1) * (l + 2), 0)))
                offset_c = Y[:, :nst] @ (supertranslation * fac)
            elif self.dataType == sigma:
                # eth eth alpha (GHP): half of the above                         (waveform_grid.py:495-503)
                fac = _ell_factors(nst, lambda l: 0.5 * math.sqrt(max((l - 1) * l * (l + 1) * (l + 2), 0)))
                offset_c = Y[:, :nst] @ (supertranslation * fac)
            elif self.dataType in (psi0, psi1, psi2, psi3):
                # psi_n picks up the higher Weyl scalars times powers of eth u'/k (waveform_grid.py:504-550):
                #   f' = f + sum_{DT>dt} C(5-dt, 5-DT) f_DT z^(DT-dt),  z = (t - alpha) gamma k eth(v.r) - eth(alpha)
                SW1 = _sf.SWSH_grid(R, 1, ell_max_st)
                fac1 = _ell_factors((ell_max_st + 1) ** 2, lambda l: math.sqrt(l * (l + 1) / 2.0))      # eth_GHP on s = 0
                eth_alpha = SW1 @ ((1 / math.sqrt(2)) * (supertranslation * fac1))
                c1, c0 = math.sqrt(2 * math.pi / 3), math.sqrt(4 * math.pi / 3)
                v = boost_velocity
                v_modes = np.array([0.0, c1 * (v[0] + 1j * v[1]), c0 * v[2], c1 * (-v[0] + 1j * v[1])], dtype=complex)
                eth_v_dot_rhat = _sf.SWSH_grid(R, 1, 1) @ ((1 / math.sqrt(2)) * v_modes)
                self.mix_A = gamma * self.kconformal * eth_v_dot_rhat
                self.mix_C = eth_alpha
                from scipy.special import comb

                for DT in range(self.dataType + 1, psi4 + 1):
                    key = "psi{}_modes".format(DataNames[DT][-1])
                    if key not in leftover:
                        raise ValueError(
                            "\nA BMS transformation of {} requires information from {}, which "
                            "has not been supplied.".format(DataNames[self.dataType], DataNames[DT])
                        )
                    w_temp = leftover.pop(key)
                    Yt = _sf.SWSH_grid(R, w_temp.spin_weight, w_temp.ell_max)
                    Bt, Kp, Np = pack_synthesis_matrix(Yt, w_temp.ell_min, w_temp.ell_max)
                    # the layout is what companions passed per call (run(companions=...)) must match; `data` is what
                    # run and synthesize use without them
                    self.mix.append(dict(
                        dataType=DT, spin_weight=int(w_temp.spin_weight), ell_min=int(w_temp.ell_min),
                        ell_max=int(w_temp.ell_max), coef=float(comb(5 - self.dataType, 5 - DT)), data=w_temp.data,
                        n_modes=w_temp.data.shape[1], Kpad=Kp, Ncpad=Np, d_B=torch.from_numpy(Bt).to(self.device),
                    ))
            elif self.dataType not in (psi4, hdot, news):
                warnings.warn(
                    f"\nNo BMS transformation is implemented for waveform objects of dataType '{DataNames[self.dataType]}'. "
                    "Proceeding with the transformation as if it were dataType 'Psi4'."
                )
        scale = self.kconformal**self.conformal_weight
        self.scale = scale
        self.Kpad = -(-2 * _sf.LM_total_size(self.ell_min, self.ell_max) // 16) * 16
        self.Ncpad = -(-2 * self.G // 64) * 64
        off = np.zeros(self.Ncpad)
        off[0 : 2 * self.G : 2] = offset_c.real
        off[1 : 2 * self.G : 2] = offset_c.imag
        scl = np.zeros(self.Ncpad)
        scl[0 : 2 * self.G : 2] = 1.0 if self.mix else scale     # with mixing the weight k^w is applied after the sum
        scl[1 : 2 * self.G : 2] = 1.0 if self.mix else scale
        self.n_modes_in = _sf.LM_total_size(self.ell_min, self.ell_max)
        self.n_modes_out = _sf.LM_total_size(self.out_ell_min, self.out_ell_max)

        dev = self.device
        f64 = torch.float64
        from . import ops

        Lt = max(self.ell_max, abs(s))
        seed_d, _, uv_d = ops.wigner_tables_device(Lt)
        d_R = torch.from_numpy(np.ascontiguousarray(R)).to(dev)
        self.d_B = torch.empty((self.Kpad, self.Ncpad), dtype=f64, device=dev)
        _lib.check(
            _lib.load().scrib200_swsh_pack(
                _lib.ptr(d_R), self.G, s, self.ell_min, self.ell_max, _lib.ptr(seed_d), _lib.ptr(uv_d), Lt, _lib.ptr(self.d_B),
                self.Kpad, self.Ncpad, _lib.stream_ptr(),
            ),
            "swsh_pack",
        )
        # the same table as three real planes Y_r, Y_i, Y_r + Y_i for the three-multiplication synthesis kernel
        self.npad3 = -(-self.n_modes_in // 8) * 8
        self.Gpad3 = -(-self.G // 32) * 32
        self.d_B3 = torch.empty((3, self.npad3, self.Gpad3), dtype=f64, device=dev)
        _lib.check(
            _lib.load().scrib200_swsh_pack3m(_lib.ptr(self.d_B), self.Kpad, self.Ncpad, self.n_modes_in, self.G, _lib.ptr(self.d_B3),
                                             self.npad3, self.Gpad3, _lib.stream_ptr()),
            "swsh_pack3m",
        )
        self.d_offset = torch.from_numpy(off).to(dev)
        self.d_scale = torch.from_numpy(scl).to(dev)
        if self.mix:
            self.d_unit = torch.zeros(self.Ncpad, dtype=f64, device=dev)
            self.d_unit[: 2 * self.G] = 1.0
            self.d_zero = torch.zeros(self.Ncpad, dtype=f64, device=dev)
            self.d_mixA = torch.from_numpy(np.ascontiguousarray(self.mix_A)).to(dev)
            self.d_mixC = torch.from_numpy(np.ascontiguousarray(self.mix_C)).to(dev)
            self.d_mixscale = torch.from_numpy(np.ascontiguousarray(scale)).to(dev)
        with torch.cuda.device(dev):
            self.analysis = ops.analysis(s, self.out_ell_min, self.out_ell_max, n_theta, n_phi)

    def _check_companions(self, companions, rows, host=False):
        """Check the companion fields of psi0..psi3 passed to one call: a list or tuple ordered psi(n+1)..psi4, each of
        shape `rows` + (n_modes_q,) in the layout of the psi*_modes the plan was built with - C-contiguous complex128 device
        tensors, or with `host` numpy arrays (returned as C-contiguous complex128 arrays).  Returns the list (or None);
        raises ValueError, and launches nothing."""
        if companions is None:
            return None
        name = DataNames[self.dataType]
        if not self.mix:
            raise ValueError(f"companions were passed to a plan for {name}, which mixes in no companion fields")
        want = ", ".join(DataNames[mx["dataType"]] for mx in self.mix)
        if not isinstance(companions, (list, tuple)) or len(companions) != len(self.mix):
            got = f"{len(companions)} fields" if isinstance(companions, (list, tuple)) else f"a {type(companions).__name__}"
            raise ValueError(f"{name} needs a list of {len(self.mix)} companion fields ordered {want}; got {got}")
        torch = self.torch
        index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        out = []
        for mx, c in zip(self.mix, companions):
            shape = tuple(int(r) for r in rows) + (mx["n_modes"],)
            if host:
                ok = isinstance(c, np.ndarray) and c.shape == shape and np.can_cast(c.dtype, np.complex128, "same_kind")
                kind, got = "numpy array", (f"{c.dtype} array of shape {c.shape}" if isinstance(c, np.ndarray) else type(c).__name__)
            else:
                ok = (torch.is_tensor(c) and c.is_cuda and c.device.index == index and c.dtype == torch.complex128
                      and tuple(c.shape) == shape and c.is_contiguous())
                kind = f"contiguous complex128 tensor on cuda:{index}"
                got = (f"{c.dtype} tensor of shape {tuple(c.shape)} on {c.device}{'' if c.is_contiguous() else ', not contiguous'}"
                       if torch.is_tensor(c) else type(c).__name__)
            if not ok:
                raise ValueError(
                    f"{name}: the companion field {DataNames[mx['dataType']]} (ell {mx['ell_min']}..{mx['ell_max']}, "
                    f"spin weight {mx['spin_weight']}; companions are ordered {want}) must be a {kind} of shape {shape}; "
                    f"got a {got}")
            out.append(np.ascontiguousarray(c, dtype=np.complex128) if host else c)
        return out

    def synthesize(self, data, t=None, slabs=None, companions=None):
        """[N, n_modes] complex128 -> F [N, G] complex128 (waveform_grid.py:475-559).  `t` (device) is needed for
        psi0..psi3 only, whose mixing factor depends on time.  `slabs` = [(row_lo, row_hi, event, flag), ...]: the rows of
        `data` are still arriving from the host slab by slab (ops.to_device_slabs); each slab is synthesized as soon as its
        event has fired, so the GEMM runs under the rest of the transfer.  `companions` (psi0..psi3): the higher Weyl
        scalars of this call, [N, n_modes_q] device tensors ordered psi(n+1)..psi4 (`_check_companions`); None uses the
        psi*_modes the plan was built with, uploaded on every call."""
        N = data.shape[0]
        comps = self._check_companions(companions, (N,))
        if self.mix and t is None:
            raise ValueError("TransformPlan.synthesize needs the time axis for psi0..psi3")
        return self._synthesize(data, t, slabs, self._planned_companions(N) if comps is None else comps, 1)

    def _planned_companions(self, N):
        """The psi*_modes the plan was built with as device tensors (None for a plan that mixes in none)."""
        from . import ops

        if not self.mix:
            return None
        comps = []
        for mx in self.mix:
            d = ops.to_device(mx["data"], np.complex128)
            if d.shape[0] != N:
                raise ValueError("psi*_modes must share the time axis of the waveform being transformed")
            comps.append(d)
        return comps

    def _synthesize(self, data, t, slabs, comps, n_series):
        """Synthesis of `data` [n_series * N, n_modes] (series stacked along time), then for psi0..psi3 the synthesis of each
        companion [n_series * N, n_modes_q] (the folded kernel, offset 0, scale 1) and one scrib200_weyl_mix_series launch
        that mixes them into F in place (t [N] serves every series)."""
        import ctypes

        torch = self.torch
        lib = _lib.load()
        rows = data.shape[0]
        F = torch.empty((rows, self.G), dtype=torch.complex128, device=self.device)
        cur = torch.cuda.current_stream()
        for lo, hi, ev, flag in (slabs or [(0, rows, None, None)]):
            if ev is not None:
                flag.wait()            # the copy thread has recorded the event (waiting on an unrecorded event is a no-op)
                cur.wait_event(ev)
            if hi <= lo:
                continue
            self.synthesize_with(data[lo:hi], self.d_B, self.n_modes_in, self.Kpad, self.Ncpad, self.d_offset, self.d_scale,
                                 out=F[lo:hi], d_B3=self.d_B3)
        if not self.mix:
            return F
        fields, coefs = [F], [1.0]
        for mx, d in zip(self.mix, comps):
            fields.append(self.synthesize_with(d, mx["d_B"], mx["n_modes"], mx["Kpad"], mx["Ncpad"], self.d_zero, self.d_unit,
                                               folded=True))
            coefs.append(mx["coef"])
        ptrs = (ctypes.c_void_p * len(fields))(*[f.data_ptr() for f in fields])
        cf = (ctypes.c_double * len(coefs))(*coefs)
        _lib.check(
            lib.scrib200_weyl_mix_series(
                ptrs, cf, len(fields), _lib.ptr(t), rows // n_series, n_series, self.G, _lib.ptr(self.d_alpha),
                _lib.ptr(self.d_mixA), _lib.ptr(self.d_mixC), _lib.ptr(self.d_mixscale), None, _lib.ptr(F), _lib.stream_ptr(),
            ),
            "weyl_mix_series",
        )
        return F

    # -- time-tiled remap: the layout the fused transform path hands from the remap to the analysis
    def remap_tiled(self, t, F, uprm, prep=None):
        """Same spline remap, result stored time-tiled: [ceil(N'/T), G, T] (T = self.tile)."""
        return self._remap(t, F, uprm, prep, self.tile)

    @property
    def tile(self):
        """Time-tile size of the remap -> analysis hand-off (0: tables too large, use the time-major kernels)."""
        return self.analysis.tile

    def _remap_analyze_to_host(self, t, F, uprm, prep, n_slabs):
        """Spline remap + analysis per slab of OUTPUT times, each slab's modes copied to pinned host memory on a copy stream
        while the next slab computes.  Slab boundaries are multiples of the hand-off tile; every slab is an ordinary
        scrib200_spline_remap / scrib200_map2salm_tiled call on a slice of u'."""
        torch = self.torch
        n_out = uprm.shape[0]
        host = torch.empty((n_out, self.n_modes_out), dtype=torch.complex128, pin_memory=True)
        cur = torch.cuda.current_stream()
        if self._d2h_stream is None:
            self._d2h_stream = torch.cuda.Stream()
        cs = self._d2h_stream
        per = -(-n_out // n_slabs)
        per = -(-per // self.tile) * self.tile
        for lo in range(0, n_out, per):
            hi = min(n_out, lo + per)
            modes = self.remap_analyze(t, F, uprm[lo:hi], prep, self.analysis)
            done = torch.cuda.Event()
            done.record(cur)
            cs.wait_event(done)
            with torch.cuda.stream(cs):
                host[lo:hi].copy_(modes, non_blocking=True)
            modes.record_stream(cs)
            del modes
        cs.synchronize()
        return host.numpy()

    def _run_streaming(self, t, data, slabs, t_host, debug_poison=False, on_queued=None, _speculate=True):
        """End-to-end pipeline for modes that are still arriving from the host (`slabs` of ops.to_device_slabs): slab j is
        synthesized as it lands, and every output time whose input window is already synthesized is remapped, analysed and
        copied back under the transfer of the later slabs.  Output j sits at input row lo + j; grid point g reads input
        samples at most `drift` rows away (parallel.transform_halo: alpha_g, and beta |t| / dt under a boost) and the tile
        kernel stages whole tiles plus halos, so outputs up to row r_hi - margin - lo are ready once rows < r_hi are
        synthesized (margin = drift + tile body + 2 halos + slack).  Returns (u', modes as a pinned host array) or None when
        the series is too short to be worth cutting."""
        from .parallel import SPLINE_DECAY_ROWS, transform_halo

        torch = self.torch
        lib = _lib.load()
        cur = torch.cuda.current_stream()
        # the time axis is already on the device: four tiny launches.  If this host axis was transformed before, its retained
        # block and spline halo are assumed, so the pipeline is queued without waiting for them (checked at the end)
        t_host = np.asarray(t_host, dtype=float)
        key = ("host", t_host.ctypes.data, int(t_host.shape[0]), float(t_host[0]), float(t_host[-1]), float(t_host[t_host.shape[0] // 2]))
        prep = self.prepare(t, speculate=_speculate, memo_key=key)
        lo, hi = prep.resolve()                      # host wait for those only; the modes keep streaming on the copy stream
        n_out = hi - lo
        if n_out < 8192:
            prep.verify()
            return None
        uprm = prep.uprm
        if self._d2h_stream is None:
            self._d2h_stream = torch.cuda.Stream()
        cs = self._d2h_stream
        # the output times go home first, under everything else
        u_host = torch.empty(n_out, dtype=torch.float64, pin_memory=True)
        cs.wait_stream(cur)
        with torch.cuda.stream(cs):
            u_host.copy_(uprm, non_blocking=True)
            u_landed = torch.cuda.Event()
            u_landed.record(cs)
        t_host = np.asarray(t_host, dtype=float)
        u_of_row = lambda i: (t_host[i] - self.time_translation) / self.gamma   # output time of input row i, to rounding (bounds only)
        halo, body = prep.halo_body(self.spline_halo, self.spline_body)
        drift = transform_halo(self, float(t_host[0]), float(t_host[-1]), prep.dt_min) - SPLINE_DECAY_ROWS
        margin = drift + max(body, 320) + 2 * halo + 64
        N = data.shape[0]
        # the three large intermediates live in buffers kept across calls (see _scratch): the synthesized grid, one remapped
        # slab (reused slab after slab: remap and analysis of successive slabs are ordered on this stream) and the modes
        c128 = torch.complex128
        F = _scratch("F", (N, self.G), c128, self.device)
        gridT_all = _scratch("gridT", (-(-n_out // self.tile) + 1, self.G, self.tile), c128, self.device)
        modes_all = _scratch("modes", (n_out, self.n_modes_out), c128, self.device)
        if debug_poison:
            F.fill_(float("nan"))                    # tests: an output that read a row before its synthesis turns into NaN
        host = torch.empty((n_out, self.n_modes_out), dtype=torch.complex128, pin_memory=True)
        if (n_out, self.n_modes_out) not in _spared:
            # first result of this size: leave a second page-locked block of the same size in the caching allocator, so that
            # a caller who still holds this result during the next call does not stall in cudaHostAlloc then (~90 ms)
            _spared.add((n_out, self.n_modes_out))
            del_me = torch.empty((n_out, self.n_modes_out), dtype=torch.complex128, pin_memory=True)
            del del_me
        tile = self.tile
        done = 0
        timing = ops_timing()
        for k, (rlo, rhi, ev, flag) in enumerate(slabs):
            flag.wait()
            _trace(f"slab {k} queued on the copy stream")
            cur.wait_event(ev)
            if rhi > rlo:
                self.synthesize_with(data[rlo:rhi], self.d_B, self.n_modes_in, self.Kpad, self.Ncpad, self.d_offset, self.d_scale,
                                     out=F[rlo:rhi], d_B3=self.d_B3)
            out_hi = n_out if k == len(slabs) - 1 else min(n_out, max(done, ((rhi - margin - lo) // tile) * tile))
            if out_hi > done:
                rows_needed = self.input_rows_for_outputs(t_host, u_of_row(lo + done), u_of_row(lo + out_hi - 1))
                modes = self.remap_analyze(t, F, uprm[done:out_hi], prep, self.analysis, rows_needed=rows_needed,
                                           grid_out=gridT_all[: -(-(out_hi - done) // tile)], out=modes_all[done:out_hi])
                ready = torch.cuda.Event(enable_timing=timing is not None)
                ready.record(cur)
                cs.wait_event(ready)
                with torch.cuda.stream(cs):
                    host[done:out_hi].copy_(modes, non_blocking=True)
                    if timing is not None:
                        landed = torch.cuda.Event(enable_timing=True)
                        landed.record(cs)
                        timing.append((f"outputs {done}:{out_hi} computed", ready))
                        timing.append((f"outputs {done}:{out_hi} landed on the host", landed))
                done = out_hi
        _trace("all launches queued")
        u_np, host_np = u_host.numpy(), host.numpy()         # the very objects handed to on_queued are the ones returned
        if on_queued is not None:
            # host work of the caller that can run under the pipeline: it is handed the result arrays - u' has landed, the
            # modes are still arriving - so that it can wrap them (checks on the time axis included) before the last byte
            u_landed.synchronize()
            on_queued(u_np, host_np)
        ok = prep.verify()
        cs.synchronize()
        _trace("last result slab landed")
        if not ok:                                   # the axis changed behind the same identity: once more, nothing assumed
            return self._run_streaming(t, data, slabs, t_host, debug_poison=debug_poison, _speculate=False)
        return u_np, host_np

    def run(self, t, data, return_grid=False, t_ends=None, prep=None, slabs=None, host_slabs=0, t_host=None, on_queued=None,
            companions=None):
        """Whole path on device tensors: returns (u', modes') or (u', grid' [time-major]).

        The only host round trip is the 64-byte `info` read-back (size of the retained block); it travels on a side
        stream while the synthesis kernel runs.  `prep` (from `prepare(t)`) can be reused for waveforms that share
        their time axis.  With `host_slabs` = S > 0 the modes come back as a numpy array in pinned host memory: the output
        times are cut into S slabs, each remapped, analysed and copied out on a copy stream while the next one computes
        (the end-to-end path of WaveformGrid.transform).  `companions` (psi0..psi3 only): this waveform's higher Weyl
        scalars as [N, n_modes_q] complex128 device tensors ordered psi(n+1)..psi4, in the layout of the psi*_modes the plan
        was built with; None uses those psi*_modes themselves."""
        comps = self._check_companions(companions, (data.shape[0],))
        if host_slabs and slabs is not None and t_host is not None and prep is None and self.tile and not self.mix and not return_grid:
            streamed = self._run_streaming(t, data, slabs, t_host, on_queued=on_queued)
            if streamed is not None:
                return streamed
        comps = self._planned_companions(data.shape[0]) if comps is None else comps

        def finish(F, uprm, prep):
            if return_grid:
                return self.remap(t, F, uprm, prep)
            if host_slabs and self.tile and uprm.shape[0] >= 8192:
                return self._remap_analyze_to_host(t, F, uprm, prep, host_slabs)
            return self.remap_analyze(t, F, uprm, prep, self.analysis)

        prep, out = self._step(t, data, comps, slabs=slabs, prep=prep, finish=finish)
        return prep.uprm, out

    def run_batch(self, t, data_batch, prep=None, companions=None):
        """A batch of waveforms sharing the time axis and the transformation (BASELINE config 3): data_batch
        [B, N, n_modes] device tensor -> (u' [N'], modes' [B, N', n_modes_out]).  One synthesis launch over all B*N rows,
        one spline launch with the batch in gridDim.z, one analysis launch over all B*N' rows.  psi0..psi3 need `companions`:
        each waveform's higher Weyl scalars as [B, N, n_modes_q] complex128 device tensors ordered psi(n+1)..psi4 (layout of
        the psi*_modes the plan was built with); each is synthesized over all B*N rows and one scrib200_weyl_mix_series launch
        mixes the batch."""
        B, N = int(data_batch.shape[0]), int(data_batch.shape[1])
        if t.shape[0] != N:
            raise ValueError("run_batch: the time axis must match dimension 1 of the batch")
        if self.mix and companions is None:
            raise ValueError("run_batch of psi0..psi3 needs companions=[psi(n+1), ..., psi4] as [B, N, n_modes] device tensors")
        comps = self._check_companions(companions, (B, N))
        if comps is not None:
            comps = [c.reshape(B * N, -1) for c in comps]
        prep, modes = self._step(t, data_batch.reshape(B * N, -1), comps, n_series=B, prep=prep)
        uprm = prep.uprm
        return uprm, modes.reshape(B, uprm.shape[0], -1)

    def capture(self, t, data, companions=None):
        """See CapturedTransform.  psi0..psi3 need `companions` (device tensors, as for `run`): a graph cannot contain the
        upload of the psi*_modes the plan was built with."""
        if self.mix and companions is None:
            raise ValueError("capture of psi0..psi3 needs companions=[psi(n+1), ..., psi4] as device tensors")
        self._check_companions(companions, (data.shape[0],))
        return CapturedTransform(self, t, data, companions)

    def _step(self, t, data, comps, n_series=1, slabs=None, prep=None, finish=None, capturing=False):
        """Queue one transform of `data` [n_series * N, n_modes] (series stacked along time; `slabs` as for `synthesize`)
        mixed with the psi0..psi3 companions `comps` (same stacking): the synthesis, then - unless `prep` is given - the
        preparation of `t` on the side stream under it, then `finish(F, uprm, prep)`, by default `remap_analyze`.  Returns
        (prep, out).  A time axis seen before is prepared speculatively: its retained block is assumed, so the host does
        not wait for the preparation kernels in the middle of the step (a caller streaming sub-batches would otherwise
        drain its pipeline at every one); in the rare case the kernels found another block the step is queued once more,
        unassumed.  `capturing` (a CUDA graph is being recorded): one attempt, the assumption required and verified by
        the caller after a replay."""
        torch = self.torch
        cur = torch.cuda.current_stream()
        ready = torch.cuda.Event()
        ready.record(cur)
        F = self._synthesize(data, t, slabs, comps, n_series)   # queued first: the GPU is busy while the host launches the preparation
        mine = prep is None
        for attempt in range(2):
            if mine:
                prep = self.prepare(t, overlapped=True, after=ready, speculate=(attempt == 0))
                if capturing and prep._assumed is None:
                    raise RuntimeError("CapturedTransform: the time axis must have been prepared once before the capture")
            cur.wait_event(prep.done)
            uprm = prep.uprm
            out = finish(F, uprm, prep) if finish else self.remap_analyze(t, F, uprm, prep, self.analysis, n_series)
            if capturing or not mine or prep.verify():
                return prep, out
            ready = torch.cuda.Event()            # the time axis changed behind the same storage: once more, unassumed
            ready.record(cur)


class CapturedTransform:
    """One device-resident transform (synthesis, spline preparation on its side stream, remap, analysis) recorded as a
    CUDA graph: `replay()` re-runs it on the CURRENT contents of the `t` and `data` tensors it was captured with, in one
    launch - the host is then no longer on the critical path of a step (eager, a step is ~25 launches and a few dozen
    tensor allocations; a busy or throttled host shows up as gaps between the kernels).  The retained block found when the
    graph was captured is baked into it; `verify()` checks it against what the last replay found.  For psi0..psi3 the
    graph also reads the companion tensors it was captured with (`companions`), at their contents of each replay."""

    def __init__(self, plan, t, data, companions=None):
        torch = plan.torch
        self.plan, self.t, self.data, self.companions = plan, t, data, companions
        plan.run(t, data, companions=companions)            # warms every cache the capture must not touch (memo, workspace, pinned pool)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.prep, self.modes = plan._step(t, data, companions, capturing=True)
            self.uprm = self.prep.uprm
            # the side stream (preparation + read-back of `info`) rejoins the capturing stream
            torch.cuda.current_stream().wait_stream(plan._side_stream())
        self._info_host = self.prep._host                   # the graph's read-back lands here on every replay
        self.prep._host = None

    def replay(self):
        """Queue one transform on the current stream; returns (u', modes') - the same tensors on every call."""
        self.graph.replay()
        return self.uprm, self.modes

    def verify(self):
        """After a replay has finished: is the retained block baked into the graph the one the kernels found?"""
        self.plan.torch.cuda.current_stream().synchronize()
        v = self._info_host.tolist()
        lo, hi = int(v[0]), max(int(v[0]), int(v[1]))
        return (lo, hi) == tuple(self.prep._assumed[:2])


TRACE = None        # dev aid: set to a list to collect (label, perf_counter) marks of the end-to-end pipeline


def ops_timing():
    from . import ops

    return ops.TIMING_EVENTS


def _trace(label):
    if TRACE is not None:
        import time

        TRACE.append((label, time.perf_counter()))


_plan_cache = {}
PLAN_CACHE_SIZE = 8
_spared = set()
_scratch_pool = {}


def _scratch(name, shape, dtype, device):
    """A device buffer that lives across calls (grow-only, one per name and device).  The end-to-end pipeline asks for
    the same few large intermediates on every call, interleaved on three streams; routed through the caching allocator
    the slab-sized requests found their blocks still parked behind record_stream events every few calls and fell through
    to cudaMalloc in the middle of the pipeline (5 - 95 ms stalls).  Calls on one device are serialised by their final
    synchronisation, so one buffer per role is enough."""
    import torch

    numel = 1
    for d in shape:
        numel *= int(d)
    key = (name, str(device), dtype)
    buf = _scratch_pool.get(key)
    if buf is None or buf.numel() < numel:
        _scratch_pool[key] = buf = torch.empty(max(numel, 1), dtype=dtype, device=device)
    return buf[:numel].view(*shape)


def _kwargs_key(kwargs):
    """Hashable identity of a set of transformation keywords, or None when one of them is not plain numbers (the
    psi*_modes companions of psi0..psi3 carry whole waveforms: such plans are built per call)."""
    items = []
    for k in sorted(kwargs):
        v = kwargs[k]
        if hasattr(v, "components") and not isinstance(v, np.ndarray):      # np.quaternion
            v = np.asarray(v.components, dtype=float)
        if isinstance(v, (bool, int, float, complex, np.number)):
            items.append((k, type(v).__name__, complex(v)))
            continue
        try:
            a = np.asarray(v)
        except Exception:
            return None
        if a.dtype.kind not in "biufc":
            return None
        items.append((k, a.dtype.str, a.shape, a.tobytes()))
    return tuple(items)


def cached_transform_plan(ell_min, ell_max, dataType, r_is_scaled_out=True, out_ell_max=None, **kwargs):
    """TransformPlan for this waveform layout and transformation, reused when the same transformation was planned
    before (the device tables depend on nothing else).  The plan's host algebra - rotor grid, SWSH tables of the
    supertranslation, conformal factor: ~2 ms of small numpy calls, what scri/waveform_grid.py:431-474 redoes on every
    call - is then off the critical path of every call after the first; a small LRU keeps the last few transformations."""
    torch = _lib.require_cuda()
    key = _kwargs_key(kwargs)
    if key is not None:
        key = (int(ell_min), int(ell_max), int(dataType), bool(r_is_scaled_out), out_ell_max, torch.cuda.current_device(), key)
        plan = _plan_cache.pop(key, None)
        if plan is not None:
            _plan_cache[key] = plan            # most recently used last
            return plan
    plan = TransformPlan(ell_min, ell_max, dataType, r_is_scaled_out=r_is_scaled_out, out_ell_max=out_ell_max, **kwargs)
    if key is not None and not plan.mix and not plan.leftover_kwargs:
        _plan_cache[key] = plan
        while len(_plan_cache) > PLAN_CACHE_SIZE:
            _plan_cache.pop(next(iter(_plan_cache)))
    return plan


class TimePrep:
    """Device-side products of scrib200_spline_prepare for one (plan, time axis): `tab`, `uprm_full`, `info`.

    `resolve()` waits for the 64-byte read-back and returns (lo, hi); `uprm` is the retained block u'[lo:hi]
    (scri/waveform_grid.py:564-568)."""

    def __init__(self, plan, t, overlapped=False, after=None):
        torch = plan.torch
        lib = _lib.load()
        N = t.shape[0]
        self.N = N
        self.tab = torch.empty((N, 8), dtype=torch.float64, device=plan.device)
        self.uprm_full = torch.empty(N, dtype=torch.float64, device=plan.device)
        self.info = torch.empty(8, dtype=torch.float64, device=plan.device)
        self._host = plan._info_host()
        self._pool = plan._host_pool
        cur = torch.cuda.current_stream()
        side = plan._side_stream()
        self._ready = torch.cuda.Event()
        self.done = torch.cuda.Event()

        def launch():
            _lib.check(
                lib.scrib200_spline_prepare(
                    _lib.ptr(t), N, plan.gamma if plan.divide_by_gamma else 1 / plan.gamma, int(plan.divide_by_gamma),
                    plan.time_translation, _lib.ptr(plan.d_k), _lib.ptr(plan.d_alpha), plan.G,
                    _lib.ptr(self.tab), _lib.ptr(self.uprm_full), _lib.ptr(self.info), _lib.stream_ptr(),
                ),
                "spline_prepare",
            )

        if overlapped:
            if after is not None:
                side.wait_event(after)     # t (and the tables of the plan) were ready when `after` was recorded
            else:
                side.wait_stream(cur)
            with torch.cuda.stream(side):
                launch()
                self.done.record(side)
        else:
            launch()
            self.done.record(cur)
            side.wait_stream(cur)
        # `info` is read back on the side stream so that kernels launched meanwhile on the caller's stream are not waited for
        with torch.cuda.stream(side):
            self._host.copy_(self.info, non_blocking=True)
            self._ready.record(side)
        if not torch.cuda.is_current_stream_capturing():     # (a graph's private pool keeps its tensors for the graph's lifetime)
            for x in (self.info, self.tab, self.uprm_full):
                x.record_stream(side)
        self._resolved = None
        self._assumed = None
        self._memo = None
        self._memo_key = None

    def _read_back(self):
        self._ready.synchronize()
        v = self._host.tolist()
        self._pool.append(self._host)
        self._host = None
        return (int(v[0]), max(int(v[0]), int(v[1])), float(v[2]), float(v[3]), float(v[6]))

    def resolve(self):
        if self._resolved is None:
            if self._assumed is not None:          # speculation: nothing to wait for (see GridPlan.prepare)
                self._resolved = self._assumed
            else:
                self._resolved = self._read_back()
                if self._memo is not None:
                    if len(self._memo) > 64:
                        self._memo.clear()
                    self._memo[self._memo_key] = self._resolved
            self.dt_min = self._resolved[4]        # smallest sample spacing of the time axis
        return self._resolved[:2]

    def verify(self):
        """True when the assumed retained block / decay diagnostics are what the kernels found this time (always true
        without speculation).  Waits for the read-back only - it completes right after the four preparation kernels."""
        if self._assumed is None or self._host is None:
            return True
        actual = self._read_back()
        self._memo[self._memo_key] = actual
        halo = lambda r: 32 if r[2] <= 1e-15 else (64 if r[3] <= 1e-15 else 128)
        return actual[:2] == self._assumed[:2] and halo(actual) == halo(self._assumed)

    @property
    def uprm(self):
        lo, hi = self.resolve()
        return self.uprm_full[lo:hi]

    def halo_body(self, halo=0, body=0):
        """Rows of run-in per tile side from the measured decay of the recurrences (0.268^k on uniform samples)."""
        self.resolve()
        if not halo:
            d32, d64 = self._resolved[2:4]
            halo = 32 if d32 <= 1e-15 else (64 if d64 <= 1e-15 else 128)
        return int(halo), int(body)
