"""AsymptoticBondiData / ModesTimeSeries: the Newman-Penrose scalars psi0..psi4 and the shear sigma as mode time series,
with the BMS transformation executed on the GPU.

Mirrors scri/asymptotic_bondi_data/__init__.py (container), scri/asymptotic_bondi_data/transformations.py:8-431
(`transform`: synthesis of all six fields on the boosted grid, the Horner ladders in eth u'/k, conformal weights,
per-grid-point CubicSpline remap in retarded time, spinsfast.map2salm) and scri/modes_time_series.py:72-202
(`interpolate`, time calculus, `grid_multiply`).  The per-time-step numerics run through the same C-ABI kernels as
WaveformModes.transform: scrib200_swsh_synthesize, scrib200_weyl_mix, scrib200_spline_remap, scrib200_map2salm[_tiled].
"""
import math

import numpy as np

from . import _lib, _sf, ops
from . import _quaternion as Q
from .constants import Inertial
from .plan import GridPlan, _quiet_blas, boosted_rotor_grid

# field order of the raw storage, spin weights, and the conformal weight applied by `transform`
FIELDS = ("psi0", "psi1", "psi2", "psi3", "psi4", "sigma")
SPINS = {"psi0": 2, "psi1": 1, "psi2": 0, "psi3": -1, "psi4": -2, "sigma": 2}


def _ell_array(ell_min, ell_max):
    return np.concatenate([np.full(2 * ell + 1, ell) for ell in range(ell_min, ell_max + 1)])


class ModesTimeSeries:
    """Mode weights of a spin-weighted function of time: `ndarray` [n_times, (ell_max+1)^2 - ell_min^2] complex128.

    A light stand-in for scri.ModesTimeSeries (an sf.Modes subclass, scri/modes_time_series.py): same attribute names
    (`ndarray`, `t`/`u`/`time`, `s`/`spin_weight`, `ell_min`, `ell_max`, `LM`) and the time / spin operators the hot path
    uses.  Arithmetic between series of equal layout works through `ndarray`.
    """

    __array_ufunc__ = None      # `ndarray * series` defers to __rmul__ (e.g. `abd.t * field`, bms_charges.py:165)

    def __init__(self, data, time, spin_weight, ell_max=None, ell_min=0, multiplication_truncator=max):
        self.ndarray = np.ascontiguousarray(data, dtype=complex)
        self.time = np.asarray(time, dtype=float)
        self.spin_weight = int(spin_weight)
        self.ell_min = int(ell_min)
        n = self.ndarray.shape[-1] + self.ell_min**2
        L = int(round(math.sqrt(n))) - 1
        if (L + 1) ** 2 != n or (ell_max is not None and ell_max != L):
            raise ValueError(f"mode axis of length {self.ndarray.shape[-1]} does not hold ell = {ell_min}..{ell_max}")
        self.ell_max = L
        self.multiplication_truncator = multiplication_truncator
        if self.ndarray.shape[0] != self.time.size:
            raise ValueError("first dimension of the data must match the time array")

    s = property(lambda self: self.spin_weight)
    t = property(lambda self: self.time)
    u = property(lambda self: self.time)
    n_times = property(lambda self: self.time.size)
    shape = property(lambda self: self.ndarray.shape)

    @property
    def LM(self):
        return _sf.LM_range(self.ell_min, self.ell_max)

    def _like(self, data, time=None, spin_weight=None):
        return ModesTimeSeries(data, self.time if time is None else time, self.spin_weight if spin_weight is None else spin_weight,
                               ell_min=self.ell_min, multiplication_truncator=self.multiplication_truncator)

    def copy(self):
        return self._like(self.ndarray.copy(), self.time.copy())

    def __array__(self, dtype=None, copy=None):
        return self.ndarray if dtype is None else self.ndarray.astype(dtype)

    def _aligned(self, other):
        """Both operands of a sum on a common ell range (sf.Modes zero-pads the shorter one); spin weights must agree."""
        if not isinstance(other, ModesTimeSeries):
            return self.ndarray, np.asarray(other), self
        if other.spin_weight != self.spin_weight:
            raise ValueError(f"Cannot add modes with different spin weights ({self.spin_weight} and {other.spin_weight})")
        if other.ell_min != self.ell_min:
            raise ValueError(f"Cannot add modes with different ell_min ({self.ell_min} and {other.ell_min})")
        a, b = self.ndarray, other.ndarray
        if a.shape[-1] == b.shape[-1]:
            return a, b, self
        wide, narrow = (self, other) if a.shape[-1] > b.shape[-1] else (other, self)
        padded = np.zeros(wide.ndarray.shape, dtype=complex)
        padded[..., : narrow.ndarray.shape[-1]] = narrow.ndarray
        return (a, padded, wide) if wide is self else (padded, b, wide)

    def __add__(self, other):
        a, b, like = self._aligned(other)
        return like._like(a + b, spin_weight=self.spin_weight)

    __radd__ = __add__

    def __sub__(self, other):
        a, b, like = self._aligned(other)
        return like._like(a - b, spin_weight=self.spin_weight)

    def __neg__(self):
        return self._like(-self.ndarray)

    def __mul__(self, scalar):
        if isinstance(scalar, ModesTimeSeries):      # sf.Modes `a * b` is multiply() with the object's truncator
            return self.multiply(scalar)
        if np.ndim(scalar) == 1 and np.shape(scalar)[0] == self.n_times:      # a function of time, e.g. `abd.t * field`
            scalar = np.asarray(scalar)[:, None]
        return self._like(self.ndarray * scalar)

    __rmul__ = __mul__

    def __truediv__(self, scalar):
        return self._like(self.ndarray / scalar)

    # -- spin operators (sf.Modes.eth / ethbar, NP convention; scri/modes_time_series.py:132-140 for GHP)
    def _ladder(self, sign):
        s, ell = self.spin_weight, _ell_array(self.ell_min, self.ell_max).astype(float)
        fac = np.where(ell >= abs(s), np.sqrt(np.maximum((ell - s * sign) * (ell + s * sign + 1.0), 0.0)), 0.0)
        return self._like(self.ndarray * (sign * fac)[None, :], spin_weight=s + sign)

    eth = property(lambda self: self._ladder(+1))
    ethbar = property(lambda self: self._ladder(-1))
    eth_GHP = property(lambda self: self.eth / math.sqrt(2))
    ethbar_GHP = property(lambda self: self.ethbar / math.sqrt(2))

    @property
    def bar(self):
        """Modes of the complex-conjugate function: bar(f)_{l,m} = (-1)^{s+m} conj(f_{l,-m}), spin weight -s."""
        a = self.ndarray
        out = np.empty_like(a)
        for ell in range(self.ell_min, self.ell_max + 1):      # m -> -m is a reversal inside each ell block
            i0, n = ell * ell - self.ell_min**2, 2 * ell + 1
            sign = (-1.0) ** (self.spin_weight + np.arange(-ell, ell + 1))
            np.multiply(np.conj(a[:, i0 : i0 + n][:, ::-1]), sign[None, :], out=out[:, i0 : i0 + n])
        return self._like(out, spin_weight=-self.spin_weight)

    @property
    def real(self):
        """Modes of the real part of the function (only meaningful for spin weight 0)."""
        return self._like(0.5 * (self.ndarray + self.bar.ndarray))

    # -- time calculus through the not-a-knot cubic spline (scri/modes_time_series.py:72-130)
    def interpolate(self, new_time, derivative_order=0):
        new_time = np.asarray(new_time, dtype=float)
        if new_time.ndim != 1:
            raise ValueError(f"New time array must have exactly 1 dimension; it has {new_time.ndim}.")
        if derivative_order > 3:
            raise ValueError(f"{type(self)} interpolation uses CubicSpline, and cannot take a derivative of order {derivative_order}")
        data = self.ndarray
        if derivative_order < 0:
            data = ops.spline_calculus(self.time, data, "antiderivative", -derivative_order)
        elif derivative_order in (1, 2):
            data = ops.spline_calculus(self.time, data, "derivative", derivative_order)
        elif derivative_order == 3:
            raise NotImplementedError("third derivatives are not on the GPU path")
        if derivative_order != 0 and new_time.shape == self.time.shape and np.array_equal(new_time, self.time):
            return self._like(data, new_time)
        if derivative_order != 0:
            raise NotImplementedError("derivatives are evaluated at the series' own times only")
        return self._like(ops.spline_calculus(self.time, data, "evaluate", tprime=new_time), new_time)

    def antiderivative(self, antiderivative_order=1):
        return self.interpolate(self.time, derivative_order=-antiderivative_order)

    def derivative(self, derivative_order=1):
        return self.interpolate(self.time, derivative_order=derivative_order)

    dot = property(lambda self: self.derivative())
    ddot = property(lambda self: self.derivative(2))
    int = property(lambda self: self.antiderivative())
    iint = property(lambda self: self.antiderivative(2))

    def truncate_ell(self, new_ell_max):
        n = (new_ell_max + 1) ** 2 - self.ell_min**2
        return self._like(self.ndarray[:, :n])

    def grid_multiply(self, mts, **kwargs):
        """Mode weights of the pointwise product of two functions (scri/modes_time_series.py:142-202): both are
        synthesized on the (2 L_w + 1)^2 grid (spinsfast.salm2map), multiplied, analysed (spinsfast.map2salm with
        spin s1 + s2) and truncated to `output_ell_max`.  Time is processed in slabs so the grids stay within a few GB."""
        output_ell_max = kwargs.pop("output_ell_max", self.ell_max)
        working_ell_max = kwargs.pop("working_ell_max", self.ell_max + mts.ell_max)
        if self.n_times != mts.n_times or not np.equal(self.t, mts.t).all():
            raise ValueError("The time series of objects to be multiplied must be the same.")
        n_theta = n_phi = 2 * working_ell_max + 1
        out = ops.grid_multiply(self.ndarray, self.spin_weight, self.ell_min, self.ell_max, mts.ndarray, mts.spin_weight,
                                mts.ell_min, mts.ell_max, n_theta, n_phi, working_ell_max, output_ell_max=output_ell_max)
        n_keep = (output_ell_max + 1) ** 2
        return ModesTimeSeries(out[:, :n_keep], self.t, self.spin_weight + mts.spin_weight, ell_min=0, multiplication_truncator=max)

    def multiply(self, other, truncator=None):
        """Exact product of two spin-weighted functions, truncated to ell <= truncator((ell_max1, ell_max2))
        (spherical_functions' Modes.multiply as scri/asymptotic_bondi_data/bms_charges.py:40-187 calls it; there the sum
        runs over Wigner 3j symbols).  The product of band-limited functions has band limit ell1 + ell2, for which the
        grid quadrature of `grid_multiply` is exact, so the same fused kernel is used with working_ell_max = ell1 + ell2."""
        if not isinstance(other, ModesTimeSeries):
            return self * other
        truncator = truncator or self.multiplication_truncator
        new_ell_max = int(truncator((self.ell_max, other.ell_max)))
        full = self.ell_max + other.ell_max
        keep = min(new_ell_max, full)
        out = self.grid_multiply(other, working_ell_max=full, output_ell_max=keep)
        if new_ell_max > keep:   # nothing lives above ell1 + ell2
            data = np.zeros((self.n_times, (new_ell_max + 1) ** 2), dtype=complex)
            data[:, : (keep + 1) ** 2] = out.ndarray
            out = ModesTimeSeries(data, self.t, out.spin_weight, ell_min=0, multiplication_truncator=max)
        out.multiplication_truncator = truncator
        return out


class AsymptoticBondiData:
    """psi0..psi4 and sigma as functions of retarded time, modes from ell = 0 (scri/asymptotic_bondi_data/__init__.py)."""

    def __init__(self, time, ell_max, multiplication_truncator=sum, frameType=Inertial, raw_data=None):
        self._time = np.array(time, dtype=float)
        if self._time.ndim != 1:
            raise ValueError("Input `time` parameter must be a 1-d array")
        self._ell_max = int(ell_max)
        self.frameType = frameType
        self.multiplication_truncator = multiplication_truncator
        shape = (len(FIELDS), self._time.size, (self._ell_max + 1) ** 2)
        self._raw_data = np.zeros(shape, dtype=complex) if raw_data is None else np.ascontiguousarray(raw_data, dtype=complex)
        if self._raw_data.shape != shape:
            raise ValueError(f"raw data must have shape {shape}; it has shape {self._raw_data.shape}")

    time = property(lambda self: self._time)
    t = u = time
    n_times = property(lambda self: self._time.size)
    ell_min = property(lambda self: 0)
    ell_max = property(lambda self: self._ell_max)
    n_modes = property(lambda self: (self._ell_max + 1) ** 2)

    @property
    def LM(self):
        return _sf.LM_range(0, self._ell_max)

    def _get(self, name):
        return ModesTimeSeries(self._raw_data[FIELDS.index(name)], self._time, SPINS[name], ell_min=0,
                               multiplication_truncator=self.multiplication_truncator)

    def _set(self, name, value):
        data = value.ndarray if isinstance(value, ModesTimeSeries) else np.asarray(value)
        self._raw_data[FIELDS.index(name)] = data     # broadcasts a single set of modes over time, like the reference

    def copy(self):
        return AsymptoticBondiData(self._time.copy(), self._ell_max, self.multiplication_truncator, self.frameType, self._raw_data.copy())

    @property
    def h(self):
        """The strain h = 2 bar(sigma) as a WaveformModes from ell = 2 (scri/asymptotic_bondi_data/__init__.py:120-131)."""
        from .constants import h as h_DataType
        from .waveform_modes import WaveformModes

        h_mts = 2.0 * self.sigma.bar
        s = abs(h_mts.s)
        return WaveformModes(t=h_mts.t, data=h_mts.ndarray[:, s * s :], ell_min=s, ell_max=h_mts.ell_max, frameType=Inertial,
                             dataType=h_DataType, r_is_scaled_out=True, m_is_scaled_out=True)

    def __getitem__(self, key):
        """Time slices `abd[i1:i2]` / `abd[i]` sharing the storage (scri/asymptotic_bondi_data/__init__.py:179-208)."""
        if not isinstance(key, (slice, int)):
            raise ValueError(f"Invalid key `{key}` of type `{type(key)}`.")
        if isinstance(key, int):
            key = slice(key, key + 1 if key != -1 else None)
        new = AsymptoticBondiData.__new__(AsymptoticBondiData)
        new._time = self._time[key]
        new._ell_max = self._ell_max
        new.frameType = self.frameType
        new.multiplication_truncator = self.multiplication_truncator
        new._raw_data = self._raw_data[:, key, :]
        return new

    def interpolate(self, new_times):
        new_times = np.asarray(new_times, dtype=float)
        raw = np.stack([self._get(name).interpolate(new_times).ndarray for name in FIELDS])
        return AsymptoticBondiData(new_times, self._ell_max, self.multiplication_truncator, self.frameType, raw)

    # -- BMS charges (scri/asymptotic_bondi_data/bms_charges.py); products of fields run through the fused kernel K9
    def mass_aspect(self, truncate_ell=max):
        """M = -Re{psi2 + sigma d/dt(bar sigma)} (bms_charges.py:14-47).  `truncate_ell`: a callable on (ell_max1, ell_max2)
        as in spherical_functions' Modes.multiply (default `max`), an integer (every term truncated to it), or a false value
        (the grid product with its default working band limit)."""
        if callable(truncate_ell):
            return -(self.psi2 + self.sigma.multiply(self.sigma.bar.dot, truncator=truncate_ell)).real
        if truncate_ell:
            return -(self.psi2.truncate_ell(truncate_ell) + self.sigma.multiply(self.sigma.bar.dot, truncator=lambda tup: truncate_ell)).real
        return -(self.psi2 + self.sigma * self.sigma.bar.dot).real

    @staticmethod
    def charge_vector_from_aspect(charge):
        """The ell <= 1 modes of a charge aspect as a four-vector (bms_charges.py:50-66)."""
        charge = np.asarray(charge)
        out = np.empty(charge.shape[:-1] + (4,))
        out[..., 0] = charge[..., 0].real
        out[..., 1] = (charge[..., 1] - charge[..., 3]).real / math.sqrt(6)
        out[..., 2] = (charge[..., 1] + charge[..., 3]).imag / math.sqrt(6)
        out[..., 3] = charge[..., 2].real / math.sqrt(3)
        return out / math.sqrt(4 * math.pi)

    def bondi_four_momentum(self):
        """ell < 2 part of the mass aspect as a four-vector (bms_charges.py:77-85)."""
        return self.charge_vector_from_aspect(self.mass_aspect(1).ndarray)

    def bondi_rest_mass(self):
        p = self.bondi_four_momentum()
        return np.sqrt(p[:, 0] ** 2 - np.sum(p[:, 1:] ** 2, axis=1))

    def _sigma_eth_sigma_bar(self, ell_max):
        return self.sigma.multiply(self.sigma.bar.eth_GHP, truncator=lambda tup: ell_max)

    def bondi_angular_momentum(self):
        """Total Bondi angular momentum, the ell = 1 part of i (psi1 + sigma eth(bar sigma)) (bms_charges.py:88-100; Dray 1985 eq. 8)."""
        aspect = 1j * (self.psi1.truncate_ell(1) + self._sigma_eth_sigma_bar(1)).ndarray
        return self.charge_vector_from_aspect(aspect)[:, 1:]

    def bondi_CoM_charge(self):
        """G = N + t P = -[psi1 + sigma eth(bar sigma) + eth(sigma bar sigma)/2] (bms_charges.py:173-189)."""
        aspect = -(self.psi1.truncate_ell(1) + self._sigma_eth_sigma_bar(1)
                   + 0.5 * self.sigma.multiply(self.sigma.bar, truncator=lambda tup: 1).eth_GHP).ndarray
        return self.charge_vector_from_aspect(aspect)[:, 1:]

    def bondi_boost_charge(self):
        """Bondi boost charge -[psi1 + sigma eth(bar sigma) + eth(sigma bar sigma)/2 - t eth Re{psi2 + sigma d/dt(bar sigma)}]
        (bms_charges.py:154-170)."""
        aspect = -(self.psi1.truncate_ell(1) + self._sigma_eth_sigma_bar(1)
                   + 0.5 * self.sigma.multiply(self.sigma.bar, truncator=lambda tup: 1).eth_GHP
                   - self.t * (self.psi2.truncate_ell(1) + self.sigma.multiply(self.sigma.bar.dot, truncator=lambda tup: 1)).real.eth_GHP).ndarray
        return self.charge_vector_from_aspect(aspect)[:, 1:]

    def bondi_dimensionless_spin(self):
        """Dimensionless Bondi spin vector from the boost charge, the angular momentum and the four-momentum
        (bms_charges.py:135-151)."""
        N, J, P = self.bondi_boost_charge(), self.bondi_angular_momentum(), self.bondi_four_momentum()
        M_sqr = (P[:, 0] ** 2 - np.sum(P[:, 1:] ** 2, axis=1))[:, None]
        v = P[:, 1:] / P[:, :1]
        v_norm = np.linalg.norm(v, axis=1)
        vhat = v.copy()
        moving = v_norm != 0
        vhat[moving] = v[moving] / v_norm[moving, None]
        gamma = (1 / np.sqrt(1 - v_norm**2))[:, None]
        J_dot_vhat = np.einsum("ij,ij->i", J, vhat)[:, None]
        return (gamma * (J + np.cross(v, N)) - (gamma - 1) * J_dot_vhat * vhat) / M_sqr

    def supermomentum(self, supermomentum_def, **kwargs):
        """Psi = psi2 + sigma d/dt(bar sigma) + f, with f = 0 ('Bondi-Sachs' / 'BS'), eth^2 bar sigma ('Moreschi' / 'M'),
        (eth^2 bar sigma - ethbar^2 sigma)/2 ('Geroch' / 'G') or -ethbar^2 sigma ('Geroch-Winicour' / 'GW'); with
        `integrated=True` the modes -bar(Psi) / (2 sqrt(pi)) (bms_charges.py:192-269; arXiv:1404.2475 eqs. 6-9).  Other
        keywords go to `grid_multiply` (working_ell_max, output_ell_max)."""
        integrated = kwargs.pop("integrated", False)
        base = self.psi2 + self.sigma.grid_multiply(self.sigma.bar.dot, **kwargs)
        kind = supermomentum_def.lower()
        if kind in ("bondi-sachs", "bs"):
            psi = base
        elif kind in ("moreschi", "m"):
            psi = base + self.sigma.bar.eth_GHP.eth_GHP
        elif kind in ("geroch", "g"):
            psi = base + 0.5 * (self.sigma.bar.eth_GHP.eth_GHP - self.sigma.ethbar_GHP.ethbar_GHP)
        elif kind in ("geroch-winicour", "gw"):
            psi = base - self.sigma.ethbar_GHP.ethbar_GHP
        else:
            raise ValueError(
                f"Supermomentum defintion '{supermomentum_def}' not recognized. Please choose one of the following options:\n"
                "  * 'Bondi-Sachs' or 'BS'\n  * 'Moreschi' or 'M'\n  * 'Geroch' or 'G'\n  * 'Geroch-Winicour' or 'GW'"
            )
        return -0.5 * psi.bar / math.sqrt(math.pi) if integrated else psi

    def transform(self, **kwargs):
        """BMS transformation of all six fields (scri/asymptotic_bondi_data/transformations.py:199-431)."""
        return transform(self, **kwargs)


for _name in FIELDS:
    setattr(AsymptoticBondiData, _name, property(lambda self, _n=_name: self._get(_n), lambda self, v, _n=_name: self._set(_n, v)))


def boosted_grid(frame_rotation, boost_velocity, n_theta, n_phi):
    """Rotors R_jk [n_theta, n_phi, 4] taking the z axis to the direction, in the original frame, of grid point (j, k) of
    the boosted and rotated frame (scri/asymptotic_bondi_data/transformations.py:100-147)."""
    R, _ = boosted_rotor_grid(Q.as_float_quat(frame_rotation), np.asarray(boost_velocity, dtype=float), n_theta, n_phi)
    return R.reshape(n_theta, n_phi, 4)


def conformal_factors(boost_velocity, distorted_grid_rotors):
    """k, eth(k)/k, 1/k and 1/k^3 on the grid, each [1, n_theta, n_phi] so that they broadcast against time
    (scri/asymptotic_bondi_data/transformations.py:150-196)."""
    v = np.asarray(boost_velocity, dtype=float)
    R = np.asarray(distorted_grid_rotors, dtype=float)
    gamma = 1 / math.sqrt(1 - np.dot(v, v))
    v_dot_r = (Q.rotate_z(R.reshape(-1, 4)) @ v).reshape(R.shape[:-1])[np.newaxis]
    c1, c0 = math.sqrt(2 * math.pi / 3), math.sqrt(4 * math.pi / 3)
    v_modes = np.array([0.0, c1 * (v[0] + 1j * v[1]), c0 * v[2], c1 * (-v[0] + 1j * v[1])], dtype=complex)
    eth_v_dot_r = (_sf.SWSH_grid(R.reshape(-1, 4), 1, 1) @ v_modes).reshape(R.shape[:-1])[np.newaxis]
    one_over_k = gamma * (1 - v_dot_r)
    return 1.0 / one_over_k, eth_v_dot_r / (1 - v_dot_r), one_over_k, one_over_k**3


def _process_transformation_kwargs(input_ell_max, **kwargs):
    """scri/asymptotic_bondi_data/transformations.py:8-97 (same keywords, checks and exception types)."""
    supertranslation = np.zeros((4,), dtype=complex)
    ell_max_supertranslation = 1
    if "supertranslation" in kwargs:
        supertranslation = np.array(kwargs.pop("supertranslation"), dtype=complex)
        if supertranslation.dtype != "complex" and supertranslation.size > 0:
            raise TypeError(
                "Input argument `supertranslation` should be a complex array with size>0.  "
                f"Got a {supertranslation.dtype} array of shape {supertranslation.shape}"
            )
        if supertranslation.size <= 4:
            supertranslation = np.pad(supertranslation, (0, 4 - supertranslation.size), "constant", constant_values=(0.0,))
        ell_max_supertranslation = int(np.sqrt(len(supertranslation))) - 1
        if (ell_max_supertranslation + 1) ** 2 != len(supertranslation):
            raise ValueError(
                "Input supertranslation parameter must contain modes from ell=0 up to some ell_max, including\n"
                "all relevant m modes in standard order.  Thus, it must be an array with length given by a "
                f"perfect square; its length is {len(supertranslation)}"
            )
        for ell in range(ell_max_supertranslation + 1):   # the ABD path symmetrises instead of raising
            for m in range(ell + 1):
                i_pos, i_neg = _sf.LM_index(ell, m, 0), _sf.LM_index(ell, -m, 0)
                a, b = supertranslation[i_pos], supertranslation[i_neg]
                supertranslation[i_pos] = (a + (-1.0) ** m * b.conjugate()) / 2.0
                supertranslation[i_neg] = (-1.0) ** m * supertranslation[i_pos].conjugate()
    s4pi, c1, c0 = math.sqrt(4 * math.pi), math.sqrt(2 * math.pi / 3), math.sqrt(4 * math.pi / 3)

    def vector_as_ell_1_modes(v):
        return np.array([c1 * (v[0] + 1j * v[1]), c0 * v[2], c1 * (-v[0] + 1j * v[1])], dtype=complex)

    spacetime_translation = np.zeros((4,), dtype=float)
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
            raise TypeError(f"Input argument `time_translation` should be a single float.  Got {t_trans}")
        supertranslation[0] = t_trans * s4pi
    output_ell_max = kwargs.pop("output_ell_max", input_ell_max)
    working_ell_max = kwargs.pop("working_ell_max", 2 * input_ell_max + ell_max_supertranslation)
    if working_ell_max < input_ell_max:
        raise ValueError(f"working_ell_max={working_ell_max} is too small; it must be at least ell_max={input_ell_max}")
    frame_rotation = Q.as_float_quat(np.array(kwargs.pop("frame_rotation", [1, 0, 0, 0]), dtype=float))
    if Q.qabs(frame_rotation) < 3e-16:
        raise ValueError(f"frame_rotation={frame_rotation} should be a single unit quaternion")
    frame_rotation = Q.qnormalized(frame_rotation)
    boost_velocity = np.array(kwargs.pop("boost_velocity", [0.0] * 3), dtype=float)
    beta = np.linalg.norm(boost_velocity)
    if boost_velocity.dtype != float or boost_velocity.shape != (3,) or beta >= 1.0:
        raise ValueError(f"Input boost_velocity=`{boost_velocity}` should be a 3-vector with magnitude strictly less than 1.0")
    return frame_rotation, boost_velocity, supertranslation, working_ell_max, output_ell_max


# Horner ladders of transformations.py:340-390: field' = weight * sum_q coef_q field_{n+q} z^q
_LADDERS = {
    "psi0": ((1.0, -4.0, 6.0, -4.0, 1.0), ("psi0", "psi1", "psi2", "psi3", "psi4")),
    "psi1": ((1.0, -3.0, 3.0, -1.0), ("psi1", "psi2", "psi3", "psi4")),
    "psi2": ((1.0, -2.0, 1.0), ("psi2", "psi3", "psi4")),
    "psi3": ((1.0, -1.0), ("psi3", "psi4")),
    "psi4": ((1.0,), ("psi4",)),
    "sigma": ((1.0,), ("sigma",)),
}


def transform(abd, **kwargs):
    """See AsymptoticBondiData.transform.  Host work: O(G L^2) tables; device work: 6 syntheses, 6 ladders, 6 spline
    remaps, 6 analyses."""
    torch = _lib.require_cuda()
    with _quiet_blas():
        frame_rotation, boost_velocity, supertranslation, Lw, Lout = _process_transformation_kwargs(abd.ell_max, **kwargs)
        n_theta = n_phi = 2 * Lw + 1
        beta = np.linalg.norm(boost_velocity)
        gamma = 1 / math.sqrt(1 - beta**2)
        R, _ = boosted_rotor_grid(frame_rotation, boost_velocity, n_theta, n_phi)
        R = R.reshape(-1, 4)
        G = R.shape[0]
        nst = supertranslation.shape[0]
        Lst = int(round(math.sqrt(nst))) - 1
        ell_st = _ell_array(0, Lst).astype(float)
        alpha = (_sf.SWSH_grid(R, 0, Lst) @ supertranslation).real
        eth_alpha = _sf.SWSH_grid(R, 1, Lst) @ (supertranslation * np.sqrt(ell_st * (ell_st + 1)) / math.sqrt(2))
        ethe_alpha = _sf.SWSH_grid(R, 2, Lst) @ (0.5 * supertranslation * np.sqrt(np.maximum((ell_st - 1) * ell_st * (ell_st + 1) * (ell_st + 2), 0.0)))
        v_dot_r = Q.rotate_z(R) @ boost_velocity
        c1, c0 = math.sqrt(2 * math.pi / 3), math.sqrt(4 * math.pi / 3)
        v = boost_velocity
        v_modes = np.array([0.0, c1 * (v[0] + 1j * v[1]), c0 * v[2], c1 * (-v[0] + 1j * v[1])], dtype=complex)
        eth_v_dot_r = _sf.SWSH_grid(R, 1, 1) @ v_modes
        one_over_k = gamma * (1 - v_dot_r)
        k = 1.0 / one_over_k
        ethk_over_k = eth_v_dot_r / (1 - v_dot_r)
        # transformations.py:393: timeprime = (u - alpha_00/sqrt(4 pi)) / gamma
        plan = GridPlan("cuda", n_theta, n_phi, gamma, (supertranslation[0] / math.sqrt(4 * math.pi)).real, k, alpha, divide_by_gamma=True)
        dev = plan.device
        # the synthesis operands sY_lm(R_g) of the six spins are built and packed on the device (scrib200_swsh_pack), as in
        # TransformPlan: at ell_max = 32 the host recurrence + packing took 4 s, the kernels of the whole transform 0.1 s
        packs = {}
        analyses = {}
        n_all = (abd.ell_max + 1) ** 2
        Kpad = -(-2 * n_all // 16) * 16
        Ncpad = -(-2 * G // 64) * 64
        d_R = torch.from_numpy(np.ascontiguousarray(R)).to(dev)
        for name in FIELDS:
            s = SPINS[name]
            Lt = max(abd.ell_max, abs(s))
            seed_d, _, uv_d = ops.wigner_tables_device(Lt)
            dB = torch.empty((Kpad, Ncpad), dtype=torch.float64, device=dev)
            _lib.check(
                _lib.load().scrib200_swsh_pack(_lib.ptr(d_R), G, s, 0, abd.ell_max, _lib.ptr(seed_d), _lib.ptr(uv_d), Lt, _lib.ptr(dB), Kpad,
                                               Ncpad, _lib.stream_ptr()),
                "swsh_pack",
            )
            packs[name] = (dB, Kpad, Ncpad)
            analyses[name] = ops.analysis(s, 0, Lout, n_theta, n_phi)
    f64 = torch.float64
    d_zero = torch.zeros(Ncpad, dtype=f64, device=dev)
    d_unit = torch.zeros(Ncpad, dtype=f64, device=dev)
    d_unit[: 2 * G] = 1.0
    d_A = torch.from_numpy(np.ascontiguousarray(ethk_over_k)).to(dev)
    d_C = torch.from_numpy(np.ascontiguousarray(eth_alpha)).to(dev)
    d_k3 = torch.from_numpy(np.ascontiguousarray(one_over_k**3)).to(dev)
    d_k1 = torch.from_numpy(np.ascontiguousarray(one_over_k)).to(dev)
    d_off = torch.from_numpy(np.ascontiguousarray(ethe_alpha)).to(dev)

    t_d = ops.to_device(abd.u, np.float64)
    prep = plan.prepare(t_d)
    n_modes = abd.n_modes
    F = {}
    cur = torch.cuda.current_stream()
    # the six fields stream in on the copy stream (staging on a helper thread) while the synthesis of the previous one runs
    incoming = [ops.to_device_slabs(abd._raw_data[FIELDS.index(name)], np.complex128, n_slabs=1) for name in FIELDS]
    for name, (d, slabs, fut) in zip(FIELDS, incoming):
        slabs[-1][3].wait()
        cur.wait_event(slabs[-1][2])
        dB, Kpad, Ncp = packs[name]
        F[name] = plan.synthesize_with(d, dB, n_modes, Kpad, Ncp, d_zero, d_unit)
    for _, _, fut in incoming:
        fut.result()                             # surfaces a failed copy
    del incoming
    for name in FIELDS:     # ascending order: each ladder only reads fields of higher index, still untouched
        coefs, names = _LADDERS[name]
        if name == "sigma":
            plan.weyl_mix([F[n] for n in names], coefs, t_d, d_A, d_C, d_k1, d_off, F[name])
        else:
            plan.weyl_mix([F[n] for n in names], coefs, t_d, d_A, d_C, d_k3, None, F[name])
    uprm = prep.uprm
    n_out = uprm.shape[0]
    # the result lands field by field in ONE pinned host block (torch's caching host allocator reuses it between calls):
    # each D2H is a DMA at PCIe rate queued behind that field's analysis, with no second host copy
    raw_t = torch.empty((len(FIELDS), n_out, (Lout + 1) ** 2), dtype=torch.complex128, pin_memory=True)
    for name in FIELDS:
        if n_out == 0:
            break
        modes = plan.remap_analyze(t_d, F[name], uprm, prep, analyses[name])
        del F[name]
        raw_t[FIELDS.index(name)].copy_(modes, non_blocking=True)
    cur.synchronize()
    raw = raw_t.numpy()
    out = AsymptoticBondiData(ops.to_host(uprm), Lout, abd.multiplication_truncator, abd.frameType, raw)
    return out
