"""WaveformModes: SWSH-mode waveform container with the reference's method surface.

Mirrors scri/waveform_modes.py (indexing :404-455, `transform` :705-719) and the operators that
scri/__init__.py:125-150 attaches to the class.  Data live in host numpy arrays as in the reference
(t float64 [n_times], data complex128 [n_times, n_modes], frame float [n_frames, 4]); every numerical
method stages them to the GPU, runs the sm_100a kernels and copies the result back.
"""
import warnings

import numpy as np

from . import _sf
from .constants import DataNames, SpinWeights, UnknownDataType
from .waveform_base import WaveformBase, waveform_alterations


class WaveformModes(WaveformBase):
    def _init_extra(self, args, kwargs):
        if len(args) == 0:
            self.__ell_min = kwargs.pop("ell_min", 0)
            self.__ell_max = kwargs.pop("ell_max", -1)
        else:
            self.__ell_min = args[0].ell_min
            self.__ell_max = args[0].ell_max
        self.__LM = _sf.LM_range(self.__ell_min, self.__ell_max) if self.__ell_max >= self.__ell_min else np.empty((0, 2), dtype=int)

    def ensure_validity(self, alter=True, assertions=False):
        ok = super().ensure_validity(alter=alter, assertions=assertions)
        errors = []
        if self.data.size:
            if self.data.dtype != np.dtype(complex):
                if alter:
                    self.data = np.asarray(self.data, dtype=complex)
                else:
                    errors.append("`data` must be complex")
            if self.data.ndim != 2:
                errors.append(f"`data` must be two-dimensional [time, mode]; it has shape {self.data.shape}")
            elif self.data.shape[1] != _sf.LM_total_size(self.ell_min, self.ell_max):
                errors.append(
                    f"second dimension of `data` ({self.data.shape[1]}) must equal the number of modes "
                    f"for ell_min={self.ell_min}, ell_max={self.ell_max} ({_sf.LM_total_size(self.ell_min, self.ell_max)})"
                )
        if self.dataType != UnknownDataType and self.ell_max >= 0 and self.ell_min < abs(SpinWeights[self.dataType]):
            pass  # the reference only warns about this in `ensure_validity`; modes below |s| are simply zero
        if errors and assertions:
            raise ValueError("\n".join(errors))
        for e in errors:
            warnings.warn(e)
        return ok and not errors

    def _copy_kwargs(self):
        kw = super()._copy_kwargs()
        kw.update(ell_min=self.ell_min, ell_max=self.ell_max)
        return kw

    # ------------------------------------------------------------------ (ell, m) layout
    @property
    def n_modes(self):
        return self.data.shape[1]

    @property
    def ell_min(self):
        return self.__ell_min

    @property
    def ell_max(self):
        return self.__ell_max

    @property
    def ells(self):
        return self.__ell_min, self.__ell_max

    @ells.setter
    def ells(self, new):
        self.__ell_min, self.__ell_max = new
        self.__LM = _sf.LM_range(self.__ell_min, self.__ell_max)

    @property
    def LM(self):
        """Array of [ell, m] pairs in storage order (scri/waveform_modes.py:404-418)."""
        return self.__LM

    def index(self, ell, m):
        """Flat index of mode (ell, m): ell(ell+1) - ell_min^2 + m (scri/waveform_modes.py:420-455)."""
        if ell < self.ell_min or ell > self.ell_max or abs(m) > ell:
            raise ValueError(f"(ell,m)=({ell},{m}) is not contained in this waveform with ell range [{self.ell_min},{self.ell_max}]")
        return _sf.LM_index(ell, m, self.ell_min)

    def indices(self, args):
        return [self.index(ell, m) for ell, m in args]

    # ------------------------------------------------------------------ BMS transformation
    def ladder_factor(self, operations, s, ell, eth_convention="NP"):
        """Factor a sequence of eth ('+', +1, 'ð') / ethbar ('-', -1, 'ð̅') operations, applied right to left, puts on
        the spin-s mode of degree ell (scri/waveform_modes.py:478-520)."""
        op_dict = {"ð": +1, "ð̅": -1, "+": +1, "-": -1, +1: +1, -1: -1}
        conv_dict = {"NP": 1.0, "GHP": 0.5}
        if isinstance(operations, str):
            operations = operations.replace("ð̅", "-").replace("ð", "+")
        keys = op_dict.keys()
        key_strings = {key for key in keys if isinstance(key, str)}
        if not set(operations).issubset(keys):
            raise ValueError(
                "operations must be a string composed of {} or a list with elements coming from the set {}".format(key_strings, set(keys))
            )
        if eth_convention not in conv_dict:
            raise ValueError("eth_convention must be one of {}".format(set(conv_dict.keys())))
        convention_factor = conv_dict[eth_convention]
        ladder = 1.0
        sign_factor = 1.0
        for op in reversed(operations):
            sign = op_dict[op]
            sign_factor *= sign
            ladder *= (ell - s * sign) * (ell + s * sign + 1.0) if (ell >= abs(s)) else 0.0
            ladder *= convention_factor
            s += sign
        return sign_factor * np.sqrt(ladder)

    def apply_eth(self, operations, eth_convention="NP"):
        """Mode data with the spin raising / lowering operators applied (scri/waveform_modes.py:522-562): a per-ell
        scale of the columns; the (ell, m) layout is unchanged."""
        s = self.spin_weight
        fac = np.concatenate([
            np.full(2 * ell + 1, self.ladder_factor(operations, s, ell, eth_convention=eth_convention))
            for ell in range(self.ell_min, self.ell_max + 1)
        ])
        return self.data * fac[None, :]

    @property
    def eth(self):
        """Spin-raised mode data (scri/waveform_modes.py:564-567)."""
        return self.apply_eth(operations="+")

    @property
    def ethbar(self):
        """Spin-lowered mode data (scri/waveform_modes.py:569-572)."""
        return self.apply_eth(operations="-")

    @waveform_alterations
    def truncate(self, tol=1e-10):
        """Zero the bits of `data` that typically contribute less than `tol` times the norm at that instant, in place
        (scri/waveform_modes.py:457-476): tol is spread over the modes as tol / sqrt(n_modes)."""
        from . import ops

        if tol != 0.0:
            tol_per_mode = tol / np.sqrt(self.n_modes)
            self.data = ops.truncate(self.data, tol_per_mode)
        self._append_history(f"{self}.truncate(tol={tol})")

    @waveform_alterations
    def convert_to_conjugate_pairs(self):
        """Store s[l,m] = (f[l,m] + conj f[l,-m]) / sqrt 2 at m > 0 and d[l,m] = (f[l,m] - conj f[l,-m]) / sqrt 2 at -m, in
        place (scri/waveform_modes.py:658-686)."""
        from . import ops

        self.data = ops.conjugate_pairs(self.data, self.ell_min, self.ell_max, inverse=False)
        self._append_history(f"{self}.convert_to_conjugate_pairs()")

    @waveform_alterations
    def convert_from_conjugate_pairs(self):
        """Undo `convert_to_conjugate_pairs` in place (scri/waveform_modes.py:688-703)."""
        from . import ops

        self.data = ops.conjugate_pairs(self.data, self.ell_min, self.ell_max, inverse=True)
        self._append_history(f"{self}.convert_from_conjugate_pairs()")

    def inner_product(self, b, t1=None, t2=None, allow_LM_differ=False, allow_times_differ=False):
        """<self, b> = integral from t1 to t2 of sum over modes of conj(self) b, through the not-a-knot cubic spline in time: a
        complex scalar (scri/waveform_modes.py:574-656).  Defaults: t1, t2 = the first and last time.

        The checks are those of flux.matrix_expectation_value: spin weights must match; ell ranges must match unless
        `allow_LM_differ`, which restricts both to the common range; times must match unless `allow_times_differ`, which
        interpolates both onto `flux.intersection` of the two axes.  On a common time axis the common ell range is a
        column window of each operand (no copy).  One streaming pass on the GPU (csrc/inner.cu)."""
        from . import _lib, ops
        from .flux import intersection

        if self.spin_weight != b.spin_weight:
            raise ValueError("Spin weights must match in inner_product")
        ell_min, ell_max = self.ell_min, self.ell_max
        clip = False
        if (self.ell_min != b.ell_min) or (self.ell_max != b.ell_max):
            if not allow_LM_differ:
                raise ValueError("ell_min and ell_max must match in inner_product (use allow_LM_differ=True to override)")
            ell_min, ell_max = max(self.ell_min, b.ell_min), min(self.ell_max, b.ell_max)
            if ell_min >= ell_max + 1:
                raise ValueError("Intersection of (ell,m) modes is empty.  Assuming this is not desired.")
            clip = True
        t_clip = None
        if not np.array_equal(self.t, b.t):
            if not allow_times_differ:
                raise ValueError("Time samples must match in inner_product (use allow_times_differ=True to override)")
            t_clip = intersection(self.t, b.t)
        _lib.require_cuda()
        times, A, B = self.t, self, b
        n = _sf.LM_total_size(ell_min, ell_max)
        a_cols = (ell_min**2 - A.ell_min**2, n)
        b_cols = (ell_min**2 - B.ell_min**2, n)
        if t_clip is not None:
            if clip:
                A, B = A[:, ell_min : ell_max + 1], B[:, ell_min : ell_max + 1]
                a_cols = b_cols = (0, n)
            times = t_clip
            A, B = A.interpolate(t_clip), B.interpolate(t_clip)
        w = ops.spline_integral_weights_device(times, t1, t2)
        return ops.inner_product(A.data, B.data, w, conjugate=True, a_cols=a_cols, b_cols=b_cols)

    def transform(self, **kwargs):
        """Apply a BMS transformation; returns a new WaveformModes (scri/waveform_modes.py:705-719).

        Keywords as in the reference: supertranslation, spacetime_translation, space_translation,
        time_translation, frame_rotation, boost_velocity, n_theta, n_phi, ell_max.
        """
        from .waveform_grid import WaveformGrid

        return WaveformGrid.transform(self, **kwargs)

    def to_grid(self, **kwargs):
        from .waveform_grid import WaveformGrid

        return WaveformGrid.from_modes(self, **kwargs)

    @classmethod
    def from_grid(cls, w_grid, ell_max):
        from .waveform_grid import WaveformGrid

        return WaveformGrid.to_modes(w_grid, ell_max)

    def __getitem__(self, key):
        """Subsets of the data: `w[i1:i2]` (times), `w[i1:i2, ell]` (one ell) or `w[i1:i2, ell_lo:ell_hi]` (ell_lo <= ell <
        ell_hi) - the second index addresses ell values, not data columns (scri/waveform_modes.py:953-1021); the columns
        kept are ell_lo^2 - ell_min^2 .. ell_hi'(ell_hi' + 2) + 1 - ell_min^2.  Returns a new object holding copies."""
        if isinstance(key, tuple) and len(key) == 1:
            key = key[0]
        new_ell_min, new_ell_max = self.ell_min, self.ell_max
        cols = slice(None)
        if isinstance(key, tuple) and len(key) == 2:
            tkey, lkey = key
            if isinstance(lkey, (int, np.integer)):
                if lkey < self.ell_min or lkey > self.ell_max:
                    raise ValueError(f"Requested ell value {lkey} lies outside WaveformModes object's ell range ({self.ell_min},{self.ell_max}).")
                new_ell_min = new_ell_max = int(lkey)
            elif isinstance(lkey, slice):
                if lkey.step and lkey.step != 1:
                    raise ValueError(f"Can only slice WaveformModes over contiguous ell values (step={lkey.step})")
                if not lkey.start and lkey.stop == 0:
                    new_ell_min, new_ell_max = 0, -1
                else:
                    new_ell_min = lkey.start if lkey.start else self.ell_min
                    new_ell_max = lkey.stop - 1 if lkey.stop else self.ell_max
                    if new_ell_min < self.ell_min or new_ell_max > self.ell_max:
                        raise ValueError(f"Requested ell range [{new_ell_min},{new_ell_max}] lies outside WaveformBase's ell range [{self.ell_min},{self.ell_max}].")
            else:
                raise ValueError(f"Don't know what to do with slice of type `{type(lkey)}`")
            cols = slice(0) if new_ell_max < new_ell_min else slice(new_ell_min**2 - self.ell_min**2, new_ell_max * (new_ell_max + 2) + 1 - self.ell_min**2)
        elif isinstance(key, (slice, int, np.integer)):
            tkey = key
        else:
            raise ValueError(f"Could not understand input `{key}` (of type `{type(key)}`) ")
        if isinstance(tkey, (int, np.integer)):
            tkey = slice(tkey, tkey + 1 if tkey != -1 else None)
        frame = self.frame[tkey] if self.frame.shape[0] == self.t.shape[0] else self.frame
        return type(self)(
            t=np.copy(self.t[tkey]), frame=np.copy(frame), data=np.copy(self.data[tkey, cols]), history=self.history[:],
            version_hist=self.version_hist[:], frameType=self.frameType, dataType=self.dataType, r_is_scaled_out=self.r_is_scaled_out,
            m_is_scaled_out=self.m_is_scaled_out, ell_min=new_ell_min, ell_max=new_ell_max, constructor_statement=f"{self}[{key}]",
        )

    def __repr__(self):
        rep = super().__repr__()
        rep += f"\n# ell_min={self.ell_min}, ell_max={self.ell_max}"
        return rep


def _attach_operators():
    """The reference attaches its operators onto WaveformModes in scri/__init__.py:125-150."""
    from . import rotations

    WaveformModes.rotate_decomposition_basis = rotations.rotate_decomposition_basis
    WaveformModes.rotate_physical_system = rotations.rotate_physical_system
    WaveformModes.to_inertial_frame = rotations.to_inertial_frame
    WaveformModes.to_corotating_frame = rotations.to_corotating_frame
    WaveformModes.to_coprecessing_frame = rotations.to_coprecessing_frame
    WaveformModes.get_alignment_of_decomposition_frame_to_modes = rotations.get_alignment_of_decomposition_frame_to_modes
    WaveformModes.align_decomposition_frame_to_modes = rotations.align_decomposition_frame_to_modes


_attach_operators()
