"""ctypes binding of libscrib200.so (the C ABI declared in include/scrib200.h).

There is deliberately no CPU fallback: if the shared library is missing or CUDA is unavailable the
operators raise.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libscrib200.so")

_lib = None

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_vp = ctypes.c_void_p
c_sz = ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol include/scrib200.h declares
SIGNATURES = {
    "scrib200_version": (c_int, []),
    "scrib200_last_error": (ctypes.c_char_p, []),
    "scrib200_launch_count": (c_i64, []),
    "scrib200_weyl_mix": (c_int, [c_vp, c_vp, c_int, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "scrib200_swsh_pack": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_vp]),
    "scrib200_grid_product": (c_int, [c_vp, c_vp, c_vp, c_i64, c_vp]),
    "scrib200_modes_product_max_shared_bytes": (c_sz, []),
    "scrib200_modes_product": (
        c_int,
        [c_vp, c_int, c_vp, c_int, c_i64, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_vp, c_int, c_vp, c_i64, c_vp, c_vp, c_int, c_vp],
    ),
    "scrib200_theta_synth": (c_int, [c_vp, c_int, c_i64, c_vp, c_vp, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "scrib200_theta_quad": (c_int, [c_vp, c_i64, c_vp, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "scrib200_integrate_angular_velocity": (c_int, [c_vp, c_i64, c_vp, c_vp, ctypes.c_double, ctypes.c_double, c_vp, c_vp]),
    "scrib200_xor_timeseries": (c_int, [c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_sz, c_vp]),
    "scrib200_xor_timeseries_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "scrib200_fletcher32": (c_int, [c_vp, c_i64, c_vp, c_vp]),
    "scrib200_multishuffle": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_int, c_vp]),
    "scrib200_conjugate_pairs": (c_int, [c_vp, c_i64, c_int, c_int, c_int, c_vp]),
    "scrib200_truncate": (c_int, [c_vp, c_i64, c_int, ctypes.c_double, c_vp]),
    "scrib200_h2d": (c_int, [c_vp, c_vp, c_sz, c_vp]),
    "scrib200_host_register": (c_int, [c_vp, c_sz]),
    "scrib200_host_unregister": (c_int, [c_vp]),
    "scrib200_rotate_modes": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "scrib200_rotate_modes_dmma": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "scrib200_swsh_synthesize": (c_int, [c_vp, c_i64, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_vp]),
    "scrib200_swsh_pack3m": (c_int, [c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_vp]),
    "scrib200_swsh_synthesize_3m": (c_int, [c_vp, c_i64, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_vp]),
    "scrib200_spline_prepare": (c_int, [c_vp, c_i64, ctypes.c_double, c_int, ctypes.c_double, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp]),
    "scrib200_spline_remap": (
        c_int,
        [c_vp, c_i64, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_int, c_int, c_int, c_int, c_vp, c_sz, c_vp],
    ),
    "scrib200_spline_remap_rows": (
        c_int,
        [c_vp, c_i64, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_int, c_int, c_int, c_int, c_i64, c_i64, c_vp, c_sz, c_vp],
    ),
    "scrib200_spline_remap_workspace_bytes": (c_sz, [c_i64, c_int, c_int, c_int]),
    "scrib200_map2salm_tile_size": (c_int, [c_int, c_int, c_int, c_int]),
    "scrib200_map2salm_tiled": (c_int, [c_vp, c_int, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
    "scrib200_map2salm_workspace_bytes": (c_sz, [c_i64, c_int, c_int, c_int]),
    "scrib200_spline_calculus": (c_int, [c_vp, c_i64, c_vp, c_int, c_vp, c_int, c_vp, c_vp, c_int, c_int, c_vp]),
    "scrib200_norm": (c_int, [c_vp, c_i64, c_int, c_vp, c_vp]),
    "scrib200_ll_ldt": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp]),
    "scrib200_ll_comparison": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    "scrib200_l_vector": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp]),
    "scrib200_dominant_eigenvector_workspace_bytes": (c_sz, [c_i64]),
    "scrib200_dominant_eigenvector": (c_int, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "scrib200_solve3": (c_int, [c_vp, c_vp, c_i64, ctypes.c_double, c_vp, c_vp]),
    "scrib200_sparse_expectation": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_vp]),
    "scrib200_sparse_expectation_ell": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp]),
    "scrib200_sparse_expectation_time": (c_int, [c_vp, c_vp, c_i64, c_int, c_vp, c_int, c_int, c_int, c_vp, c_int, c_vp, c_vp]),
    "scrib200_map2salm": (c_int, [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_sz, c_vp]),
    "scrib200_inner_product_workspace_bytes": (c_sz, [c_i64, c_int, c_int]),
    "scrib200_inner_product": (
        c_int,
        [c_vp, c_i64, c_int, c_i64, c_vp, c_i64, c_int, c_i64, c_i64, c_int, c_int, c_vp, c_int, c_int, c_vp, c_vp, c_sz, c_vp],
    ),
    "scrib200_inner_product_matrix_workspace_bytes": (c_sz, [c_int, c_int, c_i64, c_int]),
    "scrib200_inner_product_matrix": (c_int, [c_vp, c_int, c_i64, c_vp, c_int, c_i64, c_i64, c_int, c_vp, c_vp, c_vp, c_sz, c_vp]),
}


class Scrib200Error(RuntimeError):
    pass


def load(build_if_missing=True):
    """Load (building first if the sources are newer) and type the shared library."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        try:
            from . import build as _build

            if _build.needs_build() and os.path.exists("/usr/local/cuda/bin/nvcc"):
                _build.build()
        except Exception as exc:
            if not os.path.exists(LIB_PATH):
                raise
            import warnings

            warnings.warn(f"scri_b200: rebuilding libscrib200.so failed ({exc}); loading the existing, possibly stale, library")
    if not os.path.exists(LIB_PATH):
        raise Scrib200Error(
            f"{LIB_PATH} is missing: build it with `python -m scri_b200.build` (nvcc, sm_100a). "
            "scri_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what=""):
    if status != 0:
        msg = load().scrib200_last_error().decode()
        raise Scrib200Error(f"{what} failed ({status}): {msg}")


def launch_count():
    return int(load().scrib200_launch_count())


def require_cuda():
    import torch

    if not torch.cuda.is_available():
        raise Scrib200Error("scri_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.")
    return torch


def ptr(tensor):
    return ctypes.c_void_p(tensor.data_ptr())


def stream_ptr():
    import torch

    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
