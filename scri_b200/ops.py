"""Operator layer: numpy (host) in -> CUDA kernels through the C ABI -> numpy out.

Each function is the drop-in for one numba / third-party kernel the reference calls on the hot path
(SURVEY.md 8b).  Host arrays are staged through pinned memory; every function also accepts CUDA
tensors (then nothing is copied and a CUDA tensor is returned), which is what bench.py's
device-resident `value` uses.  No CPU fallback: without a CUDA device these raise Scrib200Error.
"""
import collections
import ctypes
import math
import os

import numpy as np

from . import _lib, _sf
from . import _quaternion as Q


def _torch():
    return _lib.require_cuda()


def is_tensor(x):
    return type(x).__module__.startswith("torch")


def to_device(x, dtype=None):
    """numpy -> CUDA tensor (no-op for CUDA tensors).

    Large arrays go through the library's pinned staging ring (scrib200_h2d): worker threads copy chunk i+1 into
    pinned memory while the copy engine drains chunk i, so the transfer runs at host-memcpy / PCIe speed instead of
    the pageable-copy path's ~10 GB/s and does not depend on the host process's BLAS / OpenMP thread pools.
    """
    torch = _torch()
    if is_tensor(x):
        return x if x.is_cuda else x.cuda()
    a = np.ascontiguousarray(x)
    if dtype is not None and a.dtype != dtype:
        a = a.astype(dtype)
    if a.nbytes < (1 << 20):
        return torch.from_numpy(a).cuda()
    out = torch.empty(a.shape, dtype=getattr(torch, a.dtype.name), device="cuda")
    lib = _lib.load()
    # an array that goes up a second time (a waveform whose fluxes, frames, ... are computed one after the other) is
    # page-locked in place and DMA'd directly from then on; the copy is then asynchronous on the current stream - every
    # operator that was handed numpy arrays synchronises before it returns numpy results, which is when the caller may
    # touch the array again
    _maybe_register(a)
    _lib.check(lib.scrib200_h2d(_lib.ptr(out), a.ctypes.data, a.nbytes, _lib.stream_ptr()), "h2d")
    return out


def to_device_nowait(x, dtype=None):
    """Small host array -> device without blocking the host: staged through page-locked memory of the caching host
    allocator and queued on the current stream (a pageable `.cuda()` is a synchronous copy of ~0.1 ms that also waits
    for whatever DMA is in flight)."""
    torch = _torch()
    if is_tensor(x):
        return x if x.is_cuda else x.cuda()
    a = np.ascontiguousarray(x)
    if dtype is not None and a.dtype != dtype:
        a = a.astype(dtype)
    h = torch.empty(a.shape, dtype=getattr(torch, a.dtype.name), pin_memory=True)
    h.numpy()[...] = a
    return h.to("cuda", non_blocking=True)


_h2d_pool = None


class _Done:
    """A finished future.  (Module level on purpose: a class defined per call is cyclic garbage that keeps whatever its
    methods close over - here a 124 MB device tensor - alive until the cycle collector gets round to it.)"""

    def __init__(self, v):
        self.v = v

    def result(self):
        return self.v


def to_device_async(x, dtype=None):
    """Start `to_device(x)` on a helper thread and return a future: the staging copy is C code that does not hold the
    GIL, so the caller can keep building host-side tables (the transformation plan) while the waveform streams in."""
    global _h2d_pool
    torch = _torch()
    if is_tensor(x) or np.asarray(x).nbytes < (1 << 20):
        return _Done(to_device(x, dtype))
    if _h2d_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _h2d_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="scrib200-h2d")
    dev = torch.cuda.current_device()
    stream = torch.cuda.current_stream()

    def work():
        with torch.cuda.device(dev), torch.cuda.stream(stream):
            return to_device(x, dtype)

    return _h2d_pool.submit(work)


_copy_streams = {}
TIMING_EVENTS = None      # dev aid: set to a list to collect (label, timing event) pairs of the transfers

# Arrays that go up more than once are page-locked in place on their second trip (scrib200_host_register), after which
# scrib200_h2d DMAs straight from them; a finalizer releases the registration when the array dies.  One-shot callers
# never pay for a registration.
_seen_hosts = {}          # (address, nbytes) -> trips so far (small: pruned as the arrays die)
_registered = {}          # (address, nbytes) -> finalizer
REGISTER_MIN_BYTES = 8 << 20
REGISTER_MAX_BYTES = 8 << 30


def _maybe_register(a):
    """Count this trip of host array `a`; page-lock it when it has been up before.  Returns True if `a` is page-locked."""
    import weakref

    if a.nbytes < REGISTER_MIN_BYTES or not a.flags.c_contiguous:
        return False
    key = (a.ctypes.data, a.nbytes)
    if key in _registered:
        return True
    trips = _seen_hosts.get(key, 0)
    owner = a if a.base is None else a.base
    if trips == 0:
        _seen_hosts[key] = 1
        try:
            weakref.finalize(owner, _seen_hosts.pop, key, None)
        except TypeError:          # owner does not support weak references: never register it
            _seen_hosts.pop(key, None)
        return False
    if sum(k[1] for k in _registered) + a.nbytes > REGISTER_MAX_BYTES:
        return False
    lib = _lib.load()
    rc = lib.scrib200_host_register(a.ctypes.data, a.nbytes)
    if rc < 0:
        return False
    ours = rc == 0                                 # 1: page-locked already (e.g. a view of a pinned torch tensor)

    def release(ptr=a.ctypes.data, k=key):
        _registered.pop(k, None)
        if not ours:
            return
        try:
            _torch().cuda.synchronize()            # no DMA may still be reading the pages
            lib.scrib200_host_unregister(ptr)
        except Exception:
            pass

    _registered[key] = weakref.finalize(owner, release)
    return True



def to_device_slabs(x, dtype=None, n_slabs=4, weights=None):
    """Start copying a large host array to the device in `n_slabs` row slabs on a dedicated copy stream (helper thread,
    GIL-free staging).  Returns (device tensor, slabs, future): slabs = [(row_lo, row_hi, event, flag)], the event of a slab
    fires when its rows have landed (the host flag says the event has been recorded); `future.result()` returns once every slab has been queued.  Consumers order their
    kernels after the slab events (TransformPlan.synthesize(slabs=...)), so compute overlaps the rest of the transfer."""
    global _h2d_pool
    torch = _torch()
    a = np.ascontiguousarray(x)
    if dtype is not None and a.dtype != dtype:
        a = a.astype(dtype)
    N = a.shape[0]
    locked = _maybe_register(a)
    dev = torch.cuda.current_device()
    if dev not in _copy_streams:
        _copy_streams[dev] = torch.cuda.Stream()
    cs = _copy_streams[dev]
    out = torch.empty(a.shape, dtype=getattr(torch, a.dtype.name), device="cuda")
    out.record_stream(cs)
    cs.wait_stream(torch.cuda.current_stream())          # the allocation (and whatever freed it before) is ordered first
    if weights is not None:      # slabs of unequal size (small first: the consumer starts early; small last: short tail)
        n_slabs = len(weights)
        cum = np.concatenate([[0.0], np.cumsum(np.asarray(weights, dtype=float))])
        bounds = [int(round(N * c / cum[-1])) for c in cum]
    else:
        bounds = [N * k // n_slabs for k in range(n_slabs + 1)]
    import threading

    # (row_lo, row_hi, CUDA event recorded once the slab's copies are queued, host flag set once that event exists:
    #  waiting on an event that has not been recorded yet is a no-op in CUDA, so consumers wait for the flag first)
    timed = TIMING_EVENTS is not None
    slabs = [(bounds[k], bounds[k + 1], torch.cuda.Event(enable_timing=timed), threading.Event()) for k in range(n_slabs)]
    lib = _lib.load()
    row_bytes = a.nbytes // max(N, 1)
    if timed:
        start = torch.cuda.Event(enable_timing=True)
        start.record(cs)
        TIMING_EVENTS.append(("h2d start", start))
        TIMING_EVENTS.extend((f"h2d slab {k} landed", sl[2]) for k, sl in enumerate(slabs))
    if locked:
        # page-locked source: every slab is one DMA queued right here - nothing for a helper thread to do, and the first
        # bytes move before the caller has done anything else
        for lo, hi, ev, flag in slabs:
            if hi > lo:
                _lib.check(
                    lib.scrib200_h2d(out.data_ptr() + lo * row_bytes, a.ctypes.data + lo * row_bytes, (hi - lo) * row_bytes,
                                     ctypes_void(cs.cuda_stream)),
                    "h2d",
                )
            ev.record(cs)
            flag.set()

        return out, slabs, _Done(out)
    if _h2d_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _h2d_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="scrib200-h2d")

    def work():
        try:
            with torch.cuda.device(dev):
                for lo, hi, ev, flag in slabs:
                    if hi > lo:
                        _lib.check(
                            lib.scrib200_h2d(out.data_ptr() + lo * row_bytes, a.ctypes.data + lo * row_bytes, (hi - lo) * row_bytes,
                                             ctypes_void(cs.cuda_stream)),
                            "h2d",
                        )
                    ev.record(cs)
                    flag.set()
        finally:
            for _, _, _, flag in slabs:      # never leave a consumer waiting if the copy failed
                flag.set()
        return out

    return out, slabs, _h2d_pool.submit(work)


def ctypes_void(v):
    import ctypes

    return ctypes.c_void_p(v)


def to_host(x):
    """CUDA tensor -> numpy.  The copy lands in pinned memory from torch's caching host allocator (DMA at full PCIe
    rate, no page-fault cost after the first call); the returned array owns that block until it is collected."""
    if not is_tensor(x):
        return x
    if not x.is_cuda:
        return x.numpy()
    torch = _torch()
    if x.numel() * x.element_size() < (1 << 20):
        return x.cpu().numpy()
    host = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
    host.copy_(x, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


_table_cache = {}


def wigner_tables_device(ell_max):
    torch = _torch()
    key = ("wig", ell_max, torch.cuda.current_device())
    if key not in _table_cache:
        seed, rec = _sf.wigner_tables(ell_max)
        uv = _sf.wigner_factor_table(ell_max)
        _table_cache[key] = tuple(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (seed, rec, uv))
    return _table_cache[key]


def delta_fragment_tables(ell_max):
    """Host (numpy) form of the operand table of scrib200_rotate_modes_dmma: for l = 0 .. ell_max the real matrices
    Delta^l = d^l(pi/2) (this package's D-matrix convention, scri_b200/_sf.py:wigner_D_matrices at Ra = Rb = cos(pi/4)) cut into
    the A fragments of mma.m8n8k4 - tiles [Kt][Mt][32 lanes] of Delta^T, then of Delta, zero padded; lane holds
    A[8 mm + lane / 4][4 kk + lane % 4].  Returns (table float64 [total], int32 offsets in doubles).  The CPU tests rebuild the
    matrices from it and run the kernel's five steps in numpy (tests/test_host.py)."""
    c = math.cos(math.pi / 4.0)
    flat = _sf.wigner_D_matrices(np.array(c + 0j), np.array(c + 0j), 0, ell_max)
    assert np.abs(flat.imag).max() == 0.0
    chunks, offsets, pos = [], np.zeros(ell_max + 1, dtype=np.int32), 0
    for ell in range(ell_max + 1):
        n = 2 * ell + 1
        delta = flat.real[_sf.D_offset(ell, 0) : _sf.D_offset(ell + 1, 0)].reshape(n, n)      # [m', mu]
        Mt, Kt = (n + 7) // 8, (n + 3) // 4
        offsets[ell] = pos
        for A in (delta.T, delta):
            pad = np.zeros((8 * Mt, 4 * Kt))
            pad[:n, :n] = A
            tiles = pad.reshape(Mt, 8, Kt, 4).transpose(2, 0, 1, 3).reshape(Kt, Mt, 32)       # [kk][mm][lane = 4 g + q]
            chunks.append(tiles.ravel())
            pos += Mt * Kt * 32
    return np.ascontiguousarray(np.concatenate(chunks)), offsets


def wigner_delta_fragments(ell_max):
    """Device copy of delta_fragment_tables(ell_max), cached per device: (device table, host int32 offsets)."""
    torch = _torch()
    key = ("delta", ell_max, torch.cuda.current_device())
    if key not in _table_cache:
        table, offsets = delta_fragment_tables(ell_max)
        _table_cache[key] = (torch.from_numpy(table).cuda(), offsets)
    return _table_cache[key]


def rotate_modes(data, R, ell_min, ell_max):
    """In-place Wigner-D rotation  a'_{lm} = sum_m' a_{lm'} D^l_{m'm}(R)  (scri/rotations.py:346-392).

    data: [n_times, n_modes] complex (numpy: rotated copy is written back into `data`; CUDA tensor: in place)
    R: one rotor [4] or a series [n_times, 4] (float) - or CUDA tensor of spinors [n_times, 2] complex.
    """
    torch = _torch()
    lib = _lib.load()
    d = to_device(data, np.complex128)
    if is_tensor(R):
        sp = R
        stride = 2 if sp.shape[0] == d.shape[0] and sp.dim() == 2 else 0
    else:
        Rf = np.asarray(R, dtype=float)
        sp_np = Q.as_spinor_array(Rf)
        stride = 2 if Rf.ndim == 2 else 0
        sp = to_device(sp_np, np.complex128)
    if ell_max <= 16 and not os.environ.get("SCRIB200_ROTATE_RECURRENCE"):
        # constant-matrix factorisation on the FP64 tensor cores
        frags, offsets = wigner_delta_fragments(ell_max)
        _lib.check(
            lib.scrib200_rotate_modes_dmma(_lib.ptr(d), d.shape[0], ell_min, ell_max, _lib.ptr(sp), stride, _lib.ptr(frags),
                                           offsets.ctypes.data, _lib.stream_ptr()),
            "rotate_modes_dmma",
        )
    else:
        # ell_max > 16: one Wigner recurrence per matrix element
        seed, rec, uv = wigner_tables_device(ell_max)
        _lib.check(
            lib.scrib200_rotate_modes(_lib.ptr(d), d.shape[0], ell_min, ell_max, _lib.ptr(sp), stride, _lib.ptr(seed), _lib.ptr(rec),
                                      _lib.ptr(uv), _lib.stream_ptr()),
            "rotate_modes",
        )
    if is_tensor(data):
        return data
    data[...] = to_host(d)
    return data


_quad_cache = {}


def _separable_analysis_tables(s, ell_min, ell_max, n_theta, n_phi):
    """Device tables of the separable map2salm: the packed phi-DFT operand e^{-i M phi_k}/n_phi for
    scrib200_swsh_synthesize over the rows (time, ring), and the quadrature tiles / fragments of scrib200_theta_quad."""
    from . import _product
    from .plan import pack_synthesis_matrix

    torch = _torch()
    key = (s, ell_min, ell_max, n_theta, n_phi, torch.cuda.current_device())
    if key not in _quad_cache:
        tb = _product.quad_tables(s, ell_min, ell_max, n_theta, n_phi)
        if not tb.fits:
            _quad_cache[key] = None
        else:
            nm = 2 * ell_max + 1
            phi = 2 * np.pi * np.arange(n_phi) / n_phi
            E = np.exp(-1j * np.arange(-ell_max, ell_max + 1)[:, None] * phi[None, :]) / n_phi      # [nm, n_phi]
            B, Kpad, Ncpad = pack_synthesis_matrix(E, 0, n_phi)
            unit = np.zeros(Ncpad)
            unit[: 2 * nm] = 1.0
            dev = {k: torch.from_numpy(getattr(tb, k)).cuda() for k in ("tiles", "wtfrag")}
            _quad_cache[key] = (tb, dev, torch.from_numpy(B).cuda(), Kpad, Ncpad, torch.from_numpy(unit).cuda(),
                                torch.zeros(Ncpad, dtype=torch.float64, device="cuda"))
    return _quad_cache[key]


def map2salm(grid, s, ell_max, n_theta=None, n_phi=None, ell_min=0, separable=None):
    """spinsfast.map2salm replacement, batched over leading axes: [..., n_theta, n_phi] -> [..., n_modes] (see `analyze`)."""
    if is_tensor(grid):
        g = grid
    else:
        g = to_device(np.asarray(grid, dtype=complex), np.complex128)
    if n_theta is None:
        n_theta, n_phi = g.shape[-2:]
    lead = g.shape[:-2] if g.dim() >= 2 and g.shape[-2:] == (n_theta, n_phi) else g.shape[:-1]
    g2 = g.reshape(-1, n_theta * n_phi)
    out = analyze(g2, analysis(s, ell_min, ell_max, n_theta, n_phi), separable).reshape(tuple(lead) + (-1,))
    return out if is_tensor(grid) else to_host(out)


Analysis = collections.namedtuple("Analysis", "s ell_min ell_max n_theta n_phi n_modes E Wt trig tile")
_analysis_cache = {}


def analysis(s, ell_min, ell_max, n_theta, n_phi):
    """The SWSH analysis of spin `s` onto ell_min..ell_max from the n_theta x n_phi grid, cached per (spin, ell range, grid,
    device): the tables E, Wt of scrib200_map2salm (scri_b200._sf.analysis_tables), `trig` = (cos, sin)(m phi_k)/n_phi for
    m = 0..ell_max of scrib200_map2salm_tiled (the +m column of E is (cos - i sin)/n_phi), and the time tile of the tiled
    kernel (scrib200_map2salm_tile_size; 0 when its tables do not fit: the time-major kernels then)."""
    torch = _torch()
    key = (s, ell_min, ell_max, n_theta, n_phi, torch.cuda.current_device())
    if key not in _analysis_cache:
        E, Wt = _sf.analysis_tables(s, ell_min, ell_max, n_theta, n_phi)
        trig = np.conj(E[:, ell_max:])
        E, Wt, trig = (torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (E, Wt, trig))
        tile = int(_lib.load().scrib200_map2salm_tile_size(n_theta, n_phi, ell_min, ell_max))
        _analysis_cache[key] = Analysis(s, ell_min, ell_max, n_theta, n_phi, _sf.LM_total_size(ell_min, ell_max), E, Wt, trig, tile)
    return _analysis_cache[key]


def analyze(grid, an, separable=None):
    """Analysis `an` of a time-major device grid [N, n_theta * n_phi] complex128 -> [N, an.n_modes].  From ell_max = 16 up
    it is separable on the tensor cores when its tables fit - the phi-DFT as a GEMM over the rows (time, ring), then the
    theta quadrature per M (scrib200_theta_quad); otherwise the shared-memory kernels of scrib200_map2salm.  `separable`
    True / False forces one path."""
    torch = _torch()
    lib = _lib.load()
    n_theta, n_phi, ell_max = an.n_theta, an.n_phi, an.ell_max
    sep = (_separable_analysis_tables(an.s, an.ell_min, ell_max, n_theta, n_phi)
           if (separable or (separable is None and ell_max >= 16)) else None)
    if separable and sep is None:
        raise _lib.Scrib200Error("map2salm: the separable analysis tables do not fit at this ell_max")
    N = grid.shape[0]
    if sep is not None:
        tb, dev, dB, Kpad, Ncpad, unit, zero = sep
        nm = 2 * ell_max + 1
        grid = grid.contiguous()
        P = torch.empty((N, n_theta, nm), dtype=torch.complex128, device="cuda")
        _lib.check(
            lib.scrib200_swsh_synthesize(_lib.ptr(grid), N * n_theta, n_phi, _lib.ptr(dB), Kpad, Ncpad, _lib.ptr(zero), _lib.ptr(unit), nm,
                                         _lib.ptr(P), _lib.stream_ptr()),
            "swsh_synthesize(phi-DFT)",
        )
        out = torch.empty((N, tb.n_out), dtype=torch.complex128, device="cuda")
        _lib.check(
            lib.scrib200_theta_quad(_lib.ptr(P), N, _lib.ptr(dev["tiles"]), dev["tiles"].shape[0], _lib.ptr(dev["wtfrag"]), dev["wtfrag"].shape[1],
                                    tb.cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(out), _lib.stream_ptr()),
            "theta_quad",
        )
        return out
    out = torch.empty((N, an.n_modes), dtype=torch.complex128, device=grid.device)
    need = lib.scrib200_map2salm_workspace_bytes(N, n_theta, n_phi, ell_max)
    ws = torch.empty(max(need, 16), dtype=torch.uint8, device=grid.device)
    _lib.check(
        lib.scrib200_map2salm(
            _lib.ptr(grid), N, n_theta, n_phi, _lib.ptr(an.E), _lib.ptr(an.Wt), an.ell_min, ell_max, _lib.ptr(out),
            _lib.ptr(ws), ws.numel(), _lib.stream_ptr(),
        ),
        "map2salm",
    )
    return out


_synth_cache = {}


def _regular_grid_synthesis_matrix(s, ell_min, ell_max, n_theta, n_phi):
    """Packed synthesis operand for the regular (theta, phi) grid of spinsfast (theta inclusive, phi half open)."""
    from .plan import pack_synthesis_matrix

    torch = _torch()
    key = (s, ell_min, ell_max, n_theta, n_phi, torch.cuda.current_device())
    if key not in _synth_cache:
        theta = np.linspace(0.0, np.pi, n_theta)
        phi = np.linspace(0.0, 2 * np.pi, n_phi, endpoint=False)
        th, ph = np.meshgrid(theta, phi, indexing="ij")
        R = Q.from_spherical_coords(th.ravel(), ph.ravel())
        Y = _sf.SWSH_grid(R, s, ell_max)
        B, Kpad, Ncpad = pack_synthesis_matrix(Y, ell_min, ell_max)
        unit = np.zeros(Ncpad)
        unit[: 2 * n_theta * n_phi] = 1.0
        _synth_cache[key] = (torch.from_numpy(B).cuda(), Kpad, Ncpad, torch.from_numpy(unit).cuda(), torch.zeros(Ncpad, dtype=torch.float64, device="cuda"))
    return _synth_cache[key]


_theta_cache = {}


def _separable_synthesis_tables(s, ell_min, ell_max, n_theta, n_phi):
    """Device tables of the separable salm2map: theta stage (scrib200_theta_synth) and the packed phi-DFT operand
    e^{i m phi_k} for scrib200_swsh_synthesize over the rows (time, ring).  None when the theta tables do not fit."""
    from . import _product
    from .plan import pack_synthesis_matrix

    torch = _torch()
    key = (s, ell_min, ell_max, n_theta, n_phi, torch.cuda.current_device())
    if key not in _theta_cache:
        tb = _product.theta_tables(s, ell_min, ell_max, n_theta)
        if not tb.fits:
            _theta_cache[key] = None
        else:
            nm = 2 * ell_max + 1
            phi = 2 * np.pi * np.arange(n_phi) / n_phi
            E = np.exp(1j * phi[:, None] * np.arange(-ell_max, ell_max + 1)[None, :])        # [n_phi, nm]
            B, Kpad, Ncpad = pack_synthesis_matrix(E, 0, nm)
            unit = np.zeros(Ncpad)
            unit[: 2 * n_phi] = 1.0
            dev = {k: torch.from_numpy(getattr(tb, k)).cuda() for k in ("perm", "ctl", "lamfrag")}
            _theta_cache[key] = (tb, dev, torch.from_numpy(B).cuda(), Kpad, Ncpad, torch.from_numpy(unit).cuda(),
                                 torch.zeros(Ncpad, dtype=torch.float64, device="cuda"))
    return _theta_cache[key]


def salm2map(salm, s, ell_max, n_theta, n_phi, ell_min=0, separable=None):
    """spinsfast.salm2map replacement, batched over time: [N, n_modes] -> [N, n_theta, n_phi] (device tensor in ->
    device tensor out).  From ell_max = 12 up the synthesis is separable - the Wigner-d contraction over l per ring
    (scrib200_theta_synth, FP64 DMMA) and the phi-DFT as a GEMM over the rows (time, ring); below that, or when the theta
    tables do not fit one CTA (ell_max beyond ~32), the dense synthesis GEMM (scrib200_swsh_synthesize) on the whole grid."""
    torch = _torch()
    lib = _lib.load()
    d = to_device(salm, np.complex128)
    N, G = d.shape[0], n_theta * n_phi
    sep = _separable_synthesis_tables(s, ell_min, ell_max, n_theta, n_phi) if (separable or (separable is None and ell_max >= 12)) else None
    if separable and sep is None:
        raise _lib.Scrib200Error("salm2map: the separable synthesis tables do not fit one CTA at this ell_max")
    if sep is not None:
        tb, dev, dB, Kpad, Ncpad, unit, zero = sep
        Fm = torch.empty((N, n_theta, tb.nm), dtype=torch.complex128, device="cuda")
        _lib.check(
            lib.scrib200_theta_synth(_lib.ptr(d), d.shape[1], N, _lib.ptr(dev["perm"]), _lib.ptr(dev["ctl"]), tb.n_ctl, _lib.ptr(dev["lamfrag"]),
                                     dev["lamfrag"].shape[1], tb.cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(Fm), _lib.stream_ptr()),
            "theta_synth",
        )
        F = torch.empty((N, n_theta, n_phi), dtype=torch.complex128, device="cuda")
        _lib.check(
            lib.scrib200_swsh_synthesize(_lib.ptr(Fm), N * n_theta, tb.nm, _lib.ptr(dB), Kpad, Ncpad, _lib.ptr(zero), _lib.ptr(unit), n_phi,
                                         _lib.ptr(F), _lib.stream_ptr()),
            "swsh_synthesize(phi stage)",
        )
        return F if is_tensor(salm) else to_host(F)
    dB, Kpad, Ncpad, unit, zero = _regular_grid_synthesis_matrix(s, ell_min, ell_max, n_theta, n_phi)
    F = torch.empty((N, G), dtype=torch.complex128, device="cuda")
    _lib.check(
        lib.scrib200_swsh_synthesize(_lib.ptr(d), N, d.shape[1], _lib.ptr(dB), Kpad, Ncpad, _lib.ptr(zero), _lib.ptr(unit), G, _lib.ptr(F),
                                     _lib.stream_ptr()),
        "swsh_synthesize",
    )
    F = F.reshape(N, n_theta, n_phi)
    return F if is_tensor(salm) else to_host(F)


_product_cache = {}


def _product_device_tables(key):
    torch = _torch()
    from . import _product

    dkey = key + (torch.cuda.current_device(),)
    if dkey not in _product_cache:
        tb = _product.product_tables(*key)
        dev = None
        if tb.fits:
            dev = {k: torch.from_numpy(getattr(tb, k)).cuda() for k in ("perm1", "perm2", "ctl", "lamfrag", "tiles", "wtfrag")}
        _product_cache[dkey] = (tb, dev)
    return _product_cache[dkey]


def modes_product(a, sa, a_ell_min, a_ell_max, b, sb, b_ell_min, b_ell_max, n_theta, n_phi, output_ell_max, n_ctas=0, shape=None):
    """Fused separable product (scrib200_modes_product, K9): device/host mode series in, modes of the product from
    ell = 0 to output_ell_max out; None when the problem does not fit one CTA (callers use the dense path)."""
    torch = _torch()
    lib = _lib.load()
    tb, dev = _product_device_tables((sa, a_ell_min, a_ell_max, sb, b_ell_min, b_ell_max, n_theta, n_phi, output_ell_max, shape))
    if not tb.fits:
        return None
    da = to_device(a, np.complex128)
    db = to_device(b, np.complex128)
    N = da.shape[0]
    if db.shape[0] != N:
        raise ValueError("modes_product: the two series must have the same number of time steps")
    out = torch.empty((N, tb.n_out), dtype=torch.complex128, device="cuda")
    _lib.check(
        lib.scrib200_modes_product(
            _lib.ptr(da), da.shape[1], _lib.ptr(db), db.shape[1], N, _lib.ptr(dev["perm1"]), _lib.ptr(dev["perm2"]),
            _lib.ptr(dev["ctl"]), tb.n_ctl, _lib.ptr(dev["lamfrag"]), dev["lamfrag"].shape[1],
            _lib.ptr(dev["tiles"]), tb.n_tiles_arg, _lib.ptr(dev["wtfrag"]), dev["wtfrag"].shape[1],
            tb.cfg.ctypes.data_as(ctypes.c_void_p), _lib.ptr(out), n_ctas, _lib.stream_ptr(),
        ),
        "modes_product",
    )
    return out if (is_tensor(a) or is_tensor(b)) else to_host(out)


def grid_multiply(a, sa, a_ell_min, a_ell_max, b, sb, b_ell_min, b_ell_max, n_theta, n_phi, working_ell_max, slab_bytes=2 << 30,
                  output_ell_max=None, fused=True):
    """Modes (from ell = 0 to working_ell_max, or to output_ell_max when given) of the pointwise product of two mode
    series (scri/modes_time_series.py:142-202).  Fused separable kernel when the tables fit one CTA (ell up to ~35);
    otherwise salm2map x 2 -> product -> map2salm with spin sa + sb through the dense kernels, in slabs of time."""
    torch = _torch()
    lib = _lib.load()
    N = a.shape[0]
    L_out = working_ell_max if output_ell_max is None else min(output_ell_max, working_ell_max)
    if fused:
        out = modes_product(a, sa, a_ell_min, a_ell_max, b, sb, b_ell_min, b_ell_max, n_theta, n_phi, L_out)
        if out is not None:
            return out
    G = n_theta * n_phi
    n_out = (working_ell_max + 1) ** 2
    out = np.empty((N, n_out), dtype=complex)
    slab = max(1, min(N, int(slab_bytes // (16 * G * 3))))
    for i0 in range(0, N, slab):
        i1 = min(N, i0 + slab)
        ga = salm2map(to_device(a[i0:i1], np.complex128), sa, a_ell_max, n_theta, n_phi, ell_min=a_ell_min)
        gb = salm2map(to_device(b[i0:i1], np.complex128), sb, b_ell_max, n_theta, n_phi, ell_min=b_ell_min)
        _lib.check(lib.scrib200_grid_product(_lib.ptr(ga), _lib.ptr(gb), _lib.ptr(ga), ga.numel(), _lib.stream_ptr()), "grid_product")
        del gb
        out[i0:i1] = to_host(map2salm(ga.reshape(i1 - i0, G), sa + sb, working_ell_max, n_theta, n_phi, ell_min=0))
    return out[:, : (L_out + 1) ** 2]


def norm(data):
    """sum_modes |a|^2 per time step (scri/waveform_base.py:19-35)."""
    lib = _lib.load()
    torch = _torch()
    d = to_device(data, np.complex128)
    out = torch.empty(d.shape[0], dtype=torch.float64, device="cuda")
    _lib.check(lib.scrib200_norm(_lib.ptr(d), d.shape[0], d.shape[1], _lib.ptr(out), _lib.stream_ptr()), "norm")
    return out if is_tensor(data) else to_host(out)


def conjugate_pairs(data, ell_min, ell_max, inverse=False):
    """Mode data [n_times, n_modes] to / from conjugate-pair form (scri/waveform_modes.py:658-703); returns a new array
    (a tensor for tensor input, modified in place)."""
    lib = _lib.load()
    d = to_device(data, np.complex128)
    _lib.check(lib.scrib200_conjugate_pairs(_lib.ptr(d), d.shape[0], int(ell_min), int(ell_max), int(bool(inverse)), _lib.stream_ptr()),
               "conjugate_pairs")
    return d if is_tensor(data) else to_host(d)


def truncate(data, tol_per_mode):
    """Round every time step of [n_times, ...] complex data to a multiple of 2^-floor(-log2(|row| tol_per_mode))
    (scri/waveform_modes.py:457-476)."""
    lib = _lib.load()
    d = to_device(data, np.complex128)
    n_complex = int(np.prod(d.shape[1:]))
    _lib.check(lib.scrib200_truncate(_lib.ptr(d), d.shape[0], n_complex, float(tol_per_mode), _lib.stream_ptr()), "truncate")
    return d if is_tensor(data) else to_host(d)


def _ones_zeros(n):
    torch = _torch()
    key = ("oz", n, torch.cuda.current_device())
    if key not in _table_cache:
        _table_cache[key] = (torch.ones(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.float64, device="cuda"))
    return _table_cache[key]


def spline_tables(tt):
    """(tab [N, 8], halo) for the time axis `tt` (device tensor): the shared Thomas factorisation of the not-a-knot
    moment system and the run-in length its decay calls for (scrib200_spline_prepare)."""
    lib = _lib.load()
    torch = _torch()
    N = tt.shape[0]
    tab = torch.empty((N, 8), dtype=torch.float64, device="cuda")
    info = torch.empty(8, dtype=torch.float64, device="cuda")
    _lib.check(
        lib.scrib200_spline_prepare(_lib.ptr(tt), N, 1.0, 0, 0.0, None, None, 0, _lib.ptr(tab), None, _lib.ptr(info), _lib.stream_ptr()),
        "spline_prepare",
    )
    v = info.tolist()
    halo = 32 if v[2] <= 1e-15 else (64 if v[3] <= 1e-15 else 128)
    return tab, halo


def spline_calculus(t, data, kind, order=1, tprime=None):
    """Not-a-knot cubic spline along time of every (complex) column: derivative / antiderivative at the knots, or
    evaluation at `tprime`.

    Replaces CubicSpline(t, data).derivative(k)(t) (scri/waveform_base.py:689-695), .antiderivative(k)(t) (:697-703)
    and CubicSpline(t, data)(tprime) (:964).
    """
    lib = _lib.load()
    torch = _torch()
    tt = to_device(t, np.float64)
    d = to_device(data, np.complex128)
    N = d.shape[0]
    d2 = d.reshape(N, -1)
    ncol = d2.shape[1]
    tab, halo = spline_tables(tt)
    if kind in ("derivative", "antiderivative"):
        if kind == "derivative" and order not in (1, 2) or kind == "antiderivative" and order not in (1, 2):
            raise ValueError(f"spline_calculus: order={order} is not supported for kind={kind!r}")
        code = int(order) if kind == "derivative" else -int(order)
        out = torch.empty_like(d2)
        aux = torch.empty_like(d2) if code == -2 else None
        _lib.check(
            lib.scrib200_spline_calculus(_lib.ptr(tt), N, _lib.ptr(d2), ncol, _lib.ptr(tab), code, _lib.ptr(out),
                                         _lib.ptr(aux) if aux is not None else None, halo, 0, _lib.stream_ptr()),
            "spline_calculus",
        )
        out = out.reshape(d.shape)
    elif kind == "evaluate":
        tp = to_device(tprime, np.float64)
        ones, zeros = _ones_zeros(ncol)
        out = torch.empty((tp.shape[0], ncol), dtype=torch.complex128, device="cuda")
        ws = torch.empty(lib.scrib200_spline_remap_workspace_bytes(N, ncol, halo, 0), dtype=torch.uint8, device="cuda")
        _lib.check(
            lib.scrib200_spline_remap(_lib.ptr(tt), N, _lib.ptr(d2), ncol, _lib.ptr(ones), _lib.ptr(zeros), _lib.ptr(tab),
                                      _lib.ptr(tp), tp.shape[0], _lib.ptr(out), 0, halo, 0, 1, _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr()),
            "spline_remap",
        )
        out = out.reshape((tp.shape[0],) + tuple(d.shape[1:]))
    else:
        raise NotImplementedError(f"spline_calculus kind={kind!r} is not implemented on the GPU path")
    return out if is_tensor(data) else to_host(out)


# ---------------------------------------------------------------------------------- mode_calculations
def ladder_table(ell_min, ell_max):
    """[n_modes, 5] coefficient table for scrib200_ll_ldt / scrib200_l_vector.

    Columns: ladder(l,m), ladder(l,-m), ladder(l,m+1)ladder(l,m), ladder(l,-(m-1))ladder(l,-m), m, with
    ladder(l,m) = sqrt((l-m)(l+m+1)) (sf.ladder_operator_coefficient; scri/mode_calculations.py:9) and zeros
    where the reference's `if M + 1 <= L` guards exclude the term.
    """
    import math

    def lad(l, m):
        v = (l - m) * (l + m + 1)
        return math.sqrt(v) if v > 0 else 0.0

    rows = []
    for l in range(ell_min, ell_max + 1):
        for m in range(-l, l + 1):
            rows.append([
                lad(l, m) if m + 1 <= l else 0.0,
                lad(l, -m) if m - 1 >= -l else 0.0,
                lad(l, m + 1) * lad(l, m) if m + 2 <= l else 0.0,
                lad(l, -(m - 1)) * lad(l, -m) if m - 2 >= -l else 0.0,
                float(m),
            ])
    return np.array(rows, dtype=float).reshape(-1, 5)


def _ladder_device(ell_min, ell_max):
    torch = _torch()
    key = ("lad", ell_min, ell_max, torch.cuda.current_device())
    if key not in _table_cache:
        _table_cache[key] = torch.from_numpy(ladder_table(ell_min, ell_max)).cuda()
    return _table_cache[key]


def ll_ldt(data, datadot, ell_min, ell_max):
    """(<LL> [N,3,3], <Ldt> [N,3] or None)  - scri/mode_calculations.py:14-43, 209-295."""
    lib = _lib.load()
    torch = _torch()
    d = to_device(data, np.complex128)
    dd = None if datadot is None else to_device(datadot, np.complex128)
    N, n = d.shape
    coef = _ladder_device(ell_min, ell_max)
    LL = torch.empty((N, 3, 3), dtype=torch.float64, device="cuda")
    Ldt = None if dd is None else torch.empty((N, 3), dtype=torch.float64, device="cuda")
    _lib.check(
        lib.scrib200_ll_ldt(_lib.ptr(d), None if dd is None else _lib.ptr(dd), N, n, _lib.ptr(coef), _lib.ptr(LL),
                            None if Ldt is None else _lib.ptr(Ldt), _lib.stream_ptr()),
        "ll_ldt",
    )
    if is_tensor(data):
        return LL, Ldt
    return to_host(LL), (None if Ldt is None else to_host(Ldt))


def ll_comparison(data1, data2, ell_min, ell_max):
    """<LL> between two waveforms, complex [N,3,3] - scri/mode_calculations.py:106-206."""
    lib = _lib.load()
    torch = _torch()
    d1 = to_device(data1, np.complex128)
    d2 = d1 if data2 is data1 else to_device(data2, np.complex128)
    N, n = d1.shape
    if d2.shape != d1.shape:
        raise ValueError("ll_comparison: the two waveforms must have the same shape")
    coef = _ladder_device(ell_min, ell_max)
    out = torch.empty((N, 3, 3), dtype=torch.complex128, device="cuda")
    _lib.check(lib.scrib200_ll_comparison(_lib.ptr(d1), _lib.ptr(d2), N, n, _lib.ptr(coef), _lib.ptr(out), _lib.stream_ptr()), "ll_comparison")
    return out if is_tensor(data1) else to_host(out)


def l_vector(data1, data2, ell_min, ell_max):
    """<L> complex [N,3] - scri/mode_calculations.py:60-89."""
    lib = _lib.load()
    torch = _torch()
    d1 = to_device(data1, np.complex128)
    d2 = d1 if data2 is data1 else to_device(data2, np.complex128)
    N, n = d1.shape
    coef = _ladder_device(ell_min, ell_max)
    out = torch.empty((N, 3), dtype=torch.complex128, device="cuda")
    _lib.check(lib.scrib200_l_vector(_lib.ptr(d1), _lib.ptr(d2), N, n, _lib.ptr(coef), _lib.ptr(out), _lib.stream_ptr()), "l_vector")
    return out if is_tensor(data1) else to_host(out)


def dominant_eigenvector(LL, rough_direction, rough_index):
    """Dominant principal axis of LL made continuous - np.linalg.eigh + mode_calculations.py:316-363."""
    lib = _lib.load()
    torch = _torch()
    L = to_device(LL, np.float64)
    N = L.shape[0]
    rd = rough_direction if is_tensor(rough_direction) else to_device(np.asarray(rough_direction, dtype=float), np.float64)
    out = torch.empty((N, 3), dtype=torch.float64, device="cuda")
    need = lib.scrib200_dominant_eigenvector_workspace_bytes(N)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    _lib.check(
        lib.scrib200_dominant_eigenvector(_lib.ptr(L), N, _lib.ptr(rd), int(rough_index), _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()),
        "dominant_eigenvector",
    )
    return out if is_tensor(LL) else to_host(out)


def solve3(A, b, scale=1.0):
    """scale * A^-1 b for batched 3x3 systems - np.linalg.solve at mode_calculations.py:424."""
    lib = _lib.load()
    torch = _torch()
    Ad = to_device(A, np.float64)
    bd = to_device(b, np.float64)
    x = torch.empty_like(bd)
    _lib.check(lib.scrib200_solve3(_lib.ptr(Ad), _lib.ptr(bd), Ad.shape[0], float(scale), _lib.ptr(x), _lib.stream_ptr()), "solve3")
    return x if is_tensor(A) else to_host(x)


_sparse_cache = {}


def _ell_tables(matrices, n):
    """Column-major ELL form of K COO matrices (see scrib200_sparse_expectation_ell): (rows int32, values, widths, real)."""
    rows_all, vals_all, widths = [], [], []
    real = all(not np.iscomplexobj(m[2]) or np.all(np.asarray(m[2]).imag == 0.0) for m in matrices)
    for r, c, v in matrices:
        r, c = np.asarray(r, dtype=np.int64), np.asarray(c, dtype=np.int64)
        v = np.asarray(v, dtype=complex)
        order = np.argsort(c, kind="stable")
        r, c, v = r[order], c[order], v[order]
        counts = np.bincount(c, minlength=n) if c.size else np.zeros(n, dtype=np.int64)
        W = int(counts.max()) if c.size else 0
        slot = np.arange(c.size) - np.repeat(np.cumsum(counts) - counts, counts)      # position of each entry inside its column
        er = np.full((W, n), -1, dtype=np.int32)
        ev = np.zeros((W, n), dtype=complex)
        er[slot, c] = r
        ev[slot, c] = v
        rows_all.append(er.ravel())
        vals_all.append(ev.real.ravel() if real else ev.ravel())
        widths.append(W)
    rows = np.concatenate(rows_all) if rows_all else np.zeros(0, dtype=np.int32)
    vals = np.concatenate(vals_all) if vals_all else np.zeros(0)
    if rows.size == 0:
        rows, vals = np.full(1, -1, dtype=np.int32), np.zeros(1, dtype=float if real else complex)
    return rows, vals, widths, real


XT_BUDGET_BYTES = 108 * 1024  # shared memory per CTA (mode tiles at 528 bytes per row + the block's entries): two CTAs per SM
XT_MAX_WIDTH = 4              # entries per column and matrix the kernel's unrolled walk covers


def _time_tables(matrices, n, same):
    """Tables of scrib200_sparse_expectation_time: the per-column entry table [n][K][width] and the column blocks whose rows
    of `a` (plus, when a is not b, whose own columns of b) and entries fit the shared-memory budget.  None when the
    matrices are too wide or a column's rows do not fit."""
    rows, vals, widths, real = _ell_tables(matrices, n)
    K, width = len(matrices), int(max(widths)) if widths else 0
    if width == 0 or width > XT_MAX_WIDTH:
        return None
    esize = 16 if real else 32
    slots = K * width
    er = np.full((K, width, n), -1, dtype=np.int64)
    ev = np.zeros((K, width, n), dtype=complex)
    off = 0
    for k, W in enumerate(widths):
        er[k, :W] = rows[off : off + W * n].reshape(W, n)
        ev[k, :W] = vals[off : off + W * n].reshape(W, n)
        off += W * n
    used = er >= 0
    lo = np.where(used, er, n).min(axis=(0, 1))                 # rows touched by each column (n / -1: none)
    hi = er.max(axis=(0, 1))
    empty = hi < 0
    # unused slots: value 0 on the column's lowest row (a row its window holds anyway); all-empty columns keep row -1
    fill = np.broadcast_to(np.where(empty, -1, lo), er.shape)
    er = np.where(used, er, fill)
    dt = np.dtype([("r", "<i4"), ("p", "<i4"), ("v", "<f8")]) if real else np.dtype(
        [("r", "<i4"), ("p", "<i4"), ("v", "<f8"), ("vi", "<f8"), ("q", "<f8")])
    tab = np.zeros((n, K, width), dtype=dt)
    tab["r"] = er.transpose(2, 0, 1)
    tab["v"] = ev.real.transpose(2, 0, 1)
    if not real:
        tab["vi"] = ev.imag.transpose(2, 0, 1)

    def cost(rlo, rhi, c0, c1):          # bytes of shared memory for columns [c0, c1] touching rows [rlo, rhi]
        return ((rhi + 1 - rlo) + (0 if same else c1 + 1 - c0)) * 528 + (c1 + 1 - c0) * slots * esize

    def window(c):                       # rows column c needs staged (its own row too when b is read from a's tile)
        if empty[c]:
            return (c, c) if same else None
        return (min(int(lo[c]), c), max(int(hi[c]), c)) if same else (int(lo[c]), int(hi[c]))

    def cut(budget):
        blocks, c = [], 0
        while c < n:
            w = window(c)
            if w is None:                # nothing to do for a leading empty column
                c += 1
                continue
            c0, (rlo, rhi) = c, w
            if cost(rlo, rhi, c0, c0) > budget:
                return None              # one column alone exceeds the budget
            c += 1
            while c < n:
                w = window(c)
                nlo, nhi = (rlo, rhi) if w is None else (min(rlo, w[0]), max(rhi, w[1]))
                if cost(nlo, nhi, c0, c) > budget:
                    break
                rlo, rhi = nlo, nhi
                c += 1
            blocks.append((c0, c, rlo, rhi + 1))
        return blocks

    # the kernel sizes its tiles for the tallest row window and the widest column block of ALL blocks: cut with a smaller
    # per-block budget until that total fits
    for budget in (XT_BUDGET_BYTES, 96 << 10, 84 << 10, 72 << 10, 60 << 10, 48 << 10):
        blocks = cut(budget)
        if not blocks or len(blocks) > 32:
            return None
        max_rows = max(b[3] - b[2] for b in blocks)
        max_cols = max(b[1] - b[0] for b in blocks)
        if (max_rows + (0 if same else max_cols)) * 528 + max_cols * slots * esize <= XT_BUDGET_BYTES:
            return tab, np.asarray(blocks, dtype=np.int32).ravel(), width, real
    return None


def sparse_expectation(a, b, matrices):
    """[N, K] complex: <a|M_k|b>(t) for K sparse matrices (rows, cols, vals) - scri/flux.py:40-78."""
    import ctypes

    lib = _lib.load()
    torch = _torch()
    ad = to_device(a, np.complex128)
    bd = ad if b is a else to_device(b, np.complex128)
    N, n = ad.shape
    K = len(matrices)
    # the tables are cached on the device per set of matrix objects (the generators in flux.py are lru_cached, so the
    # same objects come back call after call; the cache keeps them alive, which keeps their ids unique)
    key = (tuple(id(m) for m in matrices), n, torch.cuda.current_device(), bd is ad)
    hit = _sparse_cache.get(key)
    if hit is None:
        if len(_sparse_cache) > 64:
            _sparse_cache.clear()
        timed = _time_tables(matrices, n, bd is ad) if K <= 32 and not os.environ.get("SCRIB200_EXPECTATION_WARP") else None
        if timed is not None and timed[2] == 1 and bd is not ad:
            timed = None        # one entry per column, two arrays to stage: the warp-per-step kernels are as fast (measured)
        if timed is not None:
            tab, blocks, width, real = timed
            dev = torch.from_numpy(tab.view(np.uint8).reshape(-1)).cuda()
            _sparse_cache[key] = ("time", dev, width, real, list(matrices), blocks)
        hit = _sparse_cache.get(key)
    if hit is None:
        rows, vals, widths, real = _ell_tables(matrices, n) if K <= 32 else (None, None, [0], False)
        # matrices with several entries per column (the momentum and boost operators) go through the ELL kernel, which
        # loads b[c] once per column; with one entry per column (L_z, L_+-) the flat COO loop is the faster one (measured)
        if K <= 32 and max(widths) >= 2:
            dev = tuple(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (rows, vals))
            hit = _sparse_cache[key] = ("ell", dev, (ctypes.c_int * K)(*widths), real, list(matrices))
        else:
            rows = np.concatenate([np.asarray(m[0], dtype=np.int32) for m in matrices])
            cols = np.concatenate([np.asarray(m[1], dtype=np.int32) for m in matrices])
            vals = np.concatenate([np.asarray(m[2], dtype=complex) for m in matrices])
            seg = np.zeros(K + 1, dtype=np.int32)
            seg[1:] = np.cumsum([len(m[0]) for m in matrices])
            hit = _sparse_cache[key] = ("coo", tuple(torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in (rows, cols, vals, seg)), None, None, list(matrices))
    out = torch.empty((N, K), dtype=torch.complex128, device="cuda")
    if hit[0] == "time":
        dev, width, real, blocks = hit[1], hit[2], hit[3], hit[5]
        _lib.check(
            lib.scrib200_sparse_expectation_time(_lib.ptr(ad), _lib.ptr(bd), N, n, _lib.ptr(dev), width, K, int(not real), blocks.ctypes.data,
                                                 len(blocks) // 4, _lib.ptr(out), _lib.stream_ptr()),
            "sparse_expectation_time",
        )
    elif hit[0] == "ell":
        (dr, dv), widths, real = hit[1], hit[2], hit[3]
        _lib.check(
            lib.scrib200_sparse_expectation_ell(_lib.ptr(ad), _lib.ptr(bd), N, n, _lib.ptr(dr), _lib.ptr(dv), widths, K, int(real), _lib.ptr(out),
                                                _lib.stream_ptr()),
            "sparse_expectation_ell",
        )
    else:
        dr, dc, dv, ds = hit[1]
        _lib.check(
            lib.scrib200_sparse_expectation(_lib.ptr(ad), _lib.ptr(bd), N, n, _lib.ptr(dr), _lib.ptr(dc), _lib.ptr(dv), None, _lib.ptr(ds), K, _lib.ptr(out), _lib.stream_ptr()),
            "sparse_expectation",
        )
    return out if is_tensor(a) else to_host(out)


# ---------------------------------------------------------------------------------- inner products (csrc/inner.cu)
def _bspline_basis(knots, x, span, p):
    """[len(x), p + 1]: the nonzero degree-p B-splines B_{span-p} .. B_{span} of `knots` at the points x, where
    knots[span] <= x <= knots[span + 1] (Cox-de Boor, vectorised over the points)."""
    x = np.asarray(x, dtype=float)
    span = np.asarray(span)
    out = np.zeros((x.size, p + 1))
    out[:, 0] = 1.0
    left = np.empty((x.size, p + 1))
    right = np.empty((x.size, p + 1))
    for j in range(1, p + 1):
        left[:, j] = x - knots[span + 1 - j]
        right[:, j] = knots[span + j] - x
        saved = np.zeros(x.size)
        for r in range(j):
            temp = out[:, r] / (right[:, r + 1] + left[:, j - r])
            out[:, r] = saved + right[:, r + 1] * temp
            saved = left[:, j - r] * temp
        out[:, j] = saved
    return out


def spline_integral_weights(t, t1=None, t2=None):
    """w [N] float64 with  sum_i w_i f_i = InterpolatedUnivariateSpline(t, f, k=3).integral(t1, t2)  for every f.

    The spline is FITPACK's interpolating cubic (s = 0) on the knots [t0]*4 + t[2:N-2] + [t_{N-1}]*4, i.e. the not-a-knot
    interpolant: f = M c with the collocation matrix M[i, j] = B_j(t_i), so the integral is beta . M^-1 f with
    beta_j = integral of B_j over [t1, t2] clipped to [t0, t_{N-1}] (the spline counts as zero outside), and w = M^-T beta.
    beta comes from the antiderivative of a cubic B-spline, (k_{j+4} - k_j)/4 times the sum of the degree-4 B-splines
    from j+1 on (knots extended by one at each end); t1 > t2 gives the negative of the integral over [t2, t1].  O(N)
    host work: two points of degree-4 basis, the banded collocation matrix and one banded solve.  Defaults: t1 = t[0],
    t2 = t[-1] (quaternion.calculus.spline_definite_integral, used by scri/mode_calculations.py:534)."""
    from scipy.linalg import solve_banded

    t = np.ascontiguousarray(t, dtype=np.float64)
    N = t.size
    if t.ndim != 1 or N < 4:
        raise ValueError(f"the cubic spline integral needs at least 4 samples; got t of shape {t.shape}")
    t1 = t[0] if t1 is None else float(t1)
    t2 = t[-1] if t2 is None else float(t2)
    sign = 1.0
    lo, hi = t1, t2
    if lo > hi:
        lo, hi, sign = hi, lo, -1.0
    lo = min(max(lo, t[0]), t[-1])
    hi = min(max(hi, t[0]), t[-1])
    if not lo < hi:
        return np.zeros(N)
    k = np.concatenate([np.full(4, t[0]), t[2 : N - 2], np.full(4, t[-1])])        # N + 4 knots, N cubic B-splines
    e = np.concatenate([[t[0]], k, [t[-1]]])                                       # N + 6 knots, N + 1 quartic ones

    def tail_sums(x):
        # S[m] = sum_{i >= m} E_i(x) for m = 0 .. N + 1 (partition of unity: 1 left of the nonzero window, 0 right of it)
        s = int(min(max(np.searchsorted(e, x, side="right") - 1, 4), N))
        vals = _bspline_basis(e, np.array([x]), np.array([s]), 4)[0]
        S = np.zeros(N + 2)
        S[: s - 4 + 1] = 1.0
        for m in range(s - 3, s + 1):
            S[m] = vals[m - (s - 4):].sum()
        return S

    c = (k[4:] - k[:N]) / 4.0
    beta = c * (tail_sums(hi)[1 : N + 1] - tail_sums(lo)[1 : N + 1])
    # collocation matrix M [N, N] with 2 bands on each side (3 kept for the last row, whose span is the last interval)
    span = np.clip(np.searchsorted(k, t, side="right") - 1, 3, N - 1)
    vals = _bspline_basis(k, t, span, 3)                                            # M[i, span_i - 3 + r]
    L = U = 3
    ab = np.zeros((L + U + 1, N))                                                   # banded form of M^T
    rows = np.arange(N)
    for r in range(4):
        j = span - 3 + r
        ab[U + j - rows, rows] = vals[:, r]                                         # M^T[j, i] = M[i, j]
    return sign * solve_banded((L, U), ab, beta)


_weights_cache = {}


def spline_integral_weights_device(t, t1=None, t2=None):
    """`spline_integral_weights` as a device tensor, cached per (t, t1, t2) on the current device."""
    torch = _torch()
    t = np.ascontiguousarray(to_host(t), dtype=np.float64)
    key = (t.tobytes(), None if t1 is None else float(t1), None if t2 is None else float(t2), torch.cuda.current_device())
    w = _weights_cache.get(key)
    if w is None:
        if len(_weights_cache) > 16:
            _weights_cache.clear()
        w = _weights_cache[key] = torch.from_numpy(spline_integral_weights(t, t1, t2)).cuda()
    return w


def _complex_device(x):
    """complex128 CUDA tensor of a host array or a tensor of any dtype."""
    torch = _torch()
    d = to_device(x, np.complex128)
    return d if d.dtype == torch.complex128 else d.to(torch.complex128)


def inner_product(a, b, w, conjugate=True, per_column=False, a_cols=None, b_cols=None):
    """Weighted sums over time of products of two complex series [N, pitch] (scrib200_inner_product):
    sum_i w_i sum_c f(a_ic) b_ic (a complex scalar tensor / numpy complex) or, with `per_column`, [n] per column;
    f = conj with `conjugate`.  `a_cols` / `b_cols` = (first column, number of columns) select a window of the rows
    (default: all columns); `w` [N] float64 (device tensor or host array)."""
    lib = _lib.load()
    torch = _torch()
    ad = _complex_device(a)
    bd = ad if b is a else _complex_device(b)
    if ad.dim() != 2 or bd.dim() != 2 or ad.shape[0] != bd.shape[0]:
        raise ValueError(f"inner_product: operands must be [N, n] with one N; got {tuple(ad.shape)} and {tuple(bd.shape)}")
    ad, bd = ad.contiguous(), bd.contiguous()
    N = ad.shape[0]
    a0, n = a_cols if a_cols is not None else (0, ad.shape[1])
    b0, nb = b_cols if b_cols is not None else (0, bd.shape[1])
    if n != nb:
        raise ValueError(f"inner_product: column windows of {n} and {nb} columns")
    wd = to_device(w, np.float64)
    if wd.shape != (N,):
        raise ValueError(f"inner_product: weights of shape {tuple(wd.shape)} for {N} samples")
    out = torch.empty(n if per_column else 1, dtype=torch.complex128, device="cuda")
    ws = torch.empty(max(16, lib.scrib200_inner_product_workspace_bytes(N, n, 1)), dtype=torch.uint8, device="cuda")
    _lib.check(
        lib.scrib200_inner_product(_lib.ptr(ad), ad.shape[1], int(a0), 0, _lib.ptr(bd), bd.shape[1], int(b0), 0, N, int(n), 1,
                                   _lib.ptr(wd), int(bool(conjugate)), int(bool(per_column)), _lib.ptr(out), _lib.ptr(ws),
                                   ws.numel(), _lib.stream_ptr()),
        "inner_product",
    )
    if not per_column:
        out = out[0]
    if is_tensor(a) or is_tensor(b):
        return out
    return to_host(out) if per_column else complex(out.item())


def _batch_operand(x):
    """[P, N, n] complex128 device tensor whose rows are contiguous within each waveform, and its waveform stride."""
    d = _complex_device(x)
    if d.dim() == 2:
        d = d.unsqueeze(0)
    if d.dim() != 3:
        raise ValueError(f"inner_product_matrix: operands must be [P, N, n]; got shape {tuple(d.shape)}")
    if d.stride(2) != 1 or d.stride(1) != d.shape[2] or d.stride(0) < d.shape[1] * d.shape[2]:
        d = d.contiguous()
    return d, d.stride(0)


def inner_product_matrix(A, B, w):
    """G [P, Q] complex128: G[p, q] = sum_i w_i sum_m conj(A[p, i, m]) B[q, i, m] (scrib200_inner_product_matrix)."""
    lib = _lib.load()
    torch = _torch()
    Ad, sa = _batch_operand(A)
    Bd, sb = (Ad, sa) if B is A else _batch_operand(B)
    P, N, n = Ad.shape
    Q = Bd.shape[0]
    if Bd.shape[1:] != (N, n):
        raise ValueError(f"inner_product_matrix: waveforms of shape {tuple(Ad.shape[1:])} and {tuple(Bd.shape[1:])}")
    wd = to_device(w, np.float64)
    if wd.shape != (N,):
        raise ValueError(f"inner_product_matrix: weights of shape {tuple(wd.shape)} for {N} samples")
    G = torch.empty((P, Q), dtype=torch.complex128, device="cuda")
    ws = torch.empty(max(16, lib.scrib200_inner_product_matrix_workspace_bytes(P, Q, N, n)), dtype=torch.uint8, device="cuda")
    _lib.check(
        lib.scrib200_inner_product_matrix(_lib.ptr(Ad), P, sa, _lib.ptr(Bd), Q, sb, N, n, _lib.ptr(wd), _lib.ptr(G), _lib.ptr(ws),
                                          ws.numel(), _lib.stream_ptr()),
        "inner_product_matrix",
    )
    return G if (is_tensor(A) or is_tensor(B)) else to_host(G)
