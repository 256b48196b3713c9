"""ctypes binding of libpcreg_b200.so (the C ABI declared in include/pcreg.h).

The library is the product: if it is missing or no CUDA device is usable, every call raises -- there
is no CPU fallback and nothing in this package imports ``oracle``.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PCREG_LIB: load another build of the same library (A/B timing of kernel variants inside one GPU session)
LIB_PATH = os.environ.get("PCREG_LIB") or os.path.join(HERE, "libpcreg_b200.so")

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_f64p = C.POINTER(C.c_double)


class PcregError(RuntimeError):
    pass


class ModelOpts(C.Structure):
    _fields_ = [("build_grid", C.c_int), ("cell_size", C.c_double), ("cells_per_point", C.c_double),
                ("max_cells", C.c_int64), ("shuffle_seed", C.c_uint64),
                ("voxel_map", C.c_int), ("voxel_scale", C.c_double), ("voxel_margin", C.c_double), ("max_voxels", C.c_int64)]


class AlignOpts(C.Structure):
    _fields_ = [("k_frac", C.c_double), ("k_abs", C.c_int64), ("R_w", C.c_double), ("r_local", C.c_double),
                ("min_local", C.c_int64), ("C1", C.c_int), ("C2", C.c_int)]


class DescOpts(C.Structure):
    _fields_ = [("min_pts", C.c_int64), ("max_pts", C.c_int64), ("R", C.c_double), ("thVar", C.c_double * 2),
                ("k_frac", C.c_double), ("align_points", C.c_int)]


class MatchOpts(C.Structure):
    _fields_ = [("unnormalize", C.c_int), ("norm_factor", C.c_double), ("change_metric", C.c_int), ("metric_factor", C.c_double),
                ("match_threshold", C.c_double), ("max_ratio", C.c_double), ("metric", C.c_int), ("unique", C.c_int)]


class RansacOpts(C.Structure):
    _fields_ = [("thDist", C.c_double), ("thInlrRatio", C.c_double), ("refine", C.c_int), ("reflection_fix", C.c_int)]


class IcpOpts(C.Structure):
    _fields_ = [("mode", C.c_int), ("iters", C.c_int), ("k_frac", C.c_double), ("R_w", C.c_double),
                ("thDist2", C.c_double), ("nn", C.c_int), ("reflection_fix", C.c_int)]


class IcpStop(C.Structure):
    _fields_ = [("tol_t", C.c_double), ("tol_r_deg", C.c_double), ("window", C.c_int)]


class IcpExtrap(C.Structure):
    _fields_ = [("angle_deg", C.c_double), ("vmax_scale", C.c_double)]


# name -> (restype, argtypes): every symbol include/pcreg.h declares
SIGNATURES = {
    "pcreg_init": (C.c_int, [c_i32p, C.c_int]),
    "pcreg_shutdown": (C.c_int, []),
    "pcreg_device_count": (C.c_int, []),
    "pcreg_last_error": (C.c_char_p, []),
    "pcreg_launch_count": (C.c_int64, []),
    "pcreg_abi_version": (C.c_int, []),
    "pcreg_model_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.POINTER(ModelOpts), C.POINTER(C.c_void_p)]),
    "pcreg_model_destroy": (C.c_int, [C.c_void_p]),
    "pcreg_model_size": (C.c_int64, [C.c_void_p]),
    "pcreg_model_grid_info": (C.c_int, [C.c_void_p, c_i32p, c_f64p, c_i64p]),
    "pcreg_model_voxel_info": (C.c_int, [C.c_void_p, c_i32p, c_f64p, c_i64p]),
    "pcreg_quick_tf": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int64, c_f64p, C.c_int, C.c_void_p, C.c_int64]),
    "pcreg_nn_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_int, c_i32p, c_f64p]),
    "pcreg_local_points_count": (C.c_int, [C.c_void_p, c_f64p, C.c_int64, C.c_int64, C.c_double, C.c_int64, C.c_int64, c_i64p, c_i32p]),
    "pcreg_local_points_fill": (C.c_int, [C.c_void_p, c_f64p, C.c_int64, C.c_int64, C.c_double, c_i64p, c_i32p, c_f64p, C.c_int64,
                                          c_f64p, c_i32p]),
    "pcreg_desc_opts_default": (None, [C.POINTER(DescOpts)]),
    "pcreg_spatial_histogram": (C.c_int, [C.c_void_p, c_f64p, C.c_int64, C.c_int64, C.POINTER(DescOpts), c_f64p, C.c_int, c_f64p, C.c_int,
                                          c_f64p, C.c_int, c_f64p, c_i32p, c_i64p]),
    "pcreg_match_opts_default": (None, [C.POINTER(MatchOpts)]),
    "pcreg_get_matches": (C.c_int, [c_f64p, C.c_int64, C.c_int64, c_f64p, C.c_int64, C.c_int64, C.c_int64, C.POINTER(MatchOpts),
                                    c_i32p, c_f64p, c_i64p]),
    "pcreg_align_opts_default": (None, [C.POINTER(AlignOpts)]),
    "pcreg_align_points": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int64, c_i64p, C.c_int64, C.POINTER(AlignOpts),
                                     C.c_void_p, c_f64p, c_f64p, c_i32p]),
    "pcreg_kabsch_batch": (C.c_int, [c_f64p, c_f64p, c_f64p, C.c_int64, c_i64p, C.c_int64, C.c_int, c_f64p, c_i32p]),
    "pcreg_ransac_score": (C.c_int, [c_f64p, c_f64p, C.c_int64, C.c_int64, c_i32p, C.c_int64, C.POINTER(RansacOpts),
                                     c_f64p, c_i32p, c_i64p, c_i64p, c_i64p, c_i64p, c_i32p, c_i32p, c_f64p]),
    "pcreg_ransac_run": (C.c_int, [c_f64p, c_f64p, C.c_int64, C.c_int64, C.c_int64, C.c_uint64, C.POINTER(RansacOpts),
                                   c_f64p, c_i32p, c_i64p, c_i64p, c_i64p, c_i64p, c_i32p]),
    "pcreg_ransac_batch": (C.c_int, [c_f64p, c_f64p, C.c_int64, c_i64p, C.c_int64, C.c_int64, c_i32p, C.POINTER(C.c_uint64),
                                     C.POINTER(RansacOpts), c_f64p, c_i32p, c_i64p, c_i64p, c_i64p, c_i64p, c_i32p]),
    "pcreg_icp_opts_default": (None, [C.POINTER(IcpOpts)]),
    "pcreg_icp_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, c_f64p, c_f64p, C.c_int64,
                                  C.POINTER(IcpOpts), c_f64p, c_f64p, c_i32p, c_i32p, c_i32p, c_f64p, c_i64p]),
    "pcreg_icp_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                      C.POINTER(IcpOpts), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcreg_icp_stop_default": (None, [C.POINTER(IcpStop)]),
    "pcreg_icp_batch_stop": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, c_f64p, c_f64p, C.c_int64,
                                       C.POINTER(IcpOpts), C.POINTER(IcpStop), c_f64p, c_f64p, c_i32p, c_i32p, c_i32p, c_f64p, c_i64p,
                                       c_i32p, c_i32p]),
    "pcreg_icp_batch_stop_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                           C.POINTER(IcpOpts), C.POINTER(IcpStop), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcreg_model_set_normals": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64]),
    "pcreg_model_compute_normals": (C.c_int, [C.c_void_p, C.c_int, c_f64p]),
    "pcreg_model_get_normals": (C.c_int, [C.c_void_p, c_f64p]),
    "pcreg_icp_batch_metric": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, c_f64p, c_f64p, C.c_int64,
                                         C.POINTER(IcpOpts), C.c_int, C.POINTER(IcpStop), c_f64p, c_f64p, c_i32p, c_i32p, c_i32p,
                                         c_f64p, c_i64p, c_i32p, c_i32p]),
    "pcreg_icp_batch_metric_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64,
                                             C.POINTER(IcpOpts), C.c_int, C.POINTER(IcpStop), C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcreg_icp_batch_gicp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int64, c_f64p, C.c_void_p, C.c_double, c_f64p,
                                       C.c_int64, C.POINTER(IcpOpts), C.POINTER(IcpStop), c_f64p, c_f64p, c_i32p, c_i32p, c_i32p, c_f64p,
                                       c_i64p, c_i32p, c_i32p]),
    "pcreg_icp_batch_gicp_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_int64,
                                           C.POINTER(IcpOpts), C.POINTER(IcpStop), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcreg_icp_batch_windows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, c_i64p, c_f64p, C.c_void_p, C.c_double, c_i64p,
                                          C.c_int64, c_f64p, C.POINTER(IcpOpts), C.c_int, C.POINTER(IcpStop), c_f64p, c_f64p, c_i32p,
                                          c_i32p, c_i32p, c_f64p, c_i64p, c_i32p, c_i32p]),
    "pcreg_icp_batch_windows_dev": (C.c_int, [C.c_void_p, C.c_void_p, c_i64p, C.c_void_p, C.c_void_p, C.c_double, c_i64p, C.c_int64,
                                              C.c_void_p, C.POINTER(IcpOpts), C.c_int, C.POINTER(IcpStop), C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p]),
    "pcreg_icp_extrap_default": (None, [C.POINTER(IcpExtrap)]),
    "pcreg_icp_batch_extrap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, c_i64p, c_f64p, c_i64p, C.c_int64, c_f64p,
                                         C.POINTER(IcpOpts), C.POINTER(IcpStop), C.POINTER(IcpExtrap), c_f64p, c_f64p, c_i32p, c_i32p,
                                         c_i32p, c_f64p, c_i64p, c_i32p, c_i32p, c_i32p]),
    "pcreg_icp_batch_extrap_dev": (C.c_int, [C.c_void_p, C.c_void_p, c_i64p, C.c_void_p, c_i64p, C.c_int64, C.c_void_p,
                                             C.POINTER(IcpOpts), C.POINTER(IcpStop), C.POINTER(IcpExtrap), C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]),
    "pcreg_icp_covariance": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, c_i64p, c_f64p, c_i64p, C.c_int64, c_f64p,
                                       C.POINTER(IcpOpts), c_f64p, c_f64p, C.c_int64, c_f64p, c_f64p, c_f64p, c_f64p, c_i32p, c_i32p,
                                       c_f64p]),
    "pcreg_icp_covariance_dev": (C.c_int, [C.c_void_p, C.c_void_p, c_i64p, C.c_void_p, c_i64p, C.c_int64, C.c_void_p,
                                           C.POINTER(IcpOpts), c_f64p, c_f64p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcreg_set_profiling": (C.c_int, [C.c_int]),
    "pcreg_last_profile": (C.c_int, [c_f64p]),
}

_lib = None
_initialised_device = None


def load():
    """dlopen the library and declare every signature.  Needs no GPU."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PcregError(
                "libpcreg_b200.so is not built (%s).  Run `python -m pcreg_b200.build` (needs nvcc). "
                "There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    msg = load().pcreg_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int, what: str) -> int:
    """Negative status -> exception; >= 0 (OK / degenerate) is returned to the caller."""
    if rc < 0:
        raise PcregError("%s failed (status %d): %s" % (what, rc, last_error()))
    return rc


def init(device=None):
    """pcreg_init on `device` -- an ordinal (default: LOCAL_RANK or 0) or a sequence of ordinals: with several devices the
    model is replicated on each and pcreg_icp_batch / pcreg_ransac_batch shard their hypotheses / windows over them inside
    the library (one host thread per device).  Raises without a usable B200."""
    global _initialised_device
    lib = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    devs = tuple(int(d) for d in device) if hasattr(device, "__len__") else (int(device),)
    if _initialised_device == devs:
        return lib
    arr = (C.c_int32 * len(devs))(*devs)
    check(lib.pcreg_init(arr, len(devs)), "pcreg_init")
    _initialised_device = devs
    return lib


def shutdown():
    global _initialised_device
    if _lib is not None:
        _lib.pcreg_shutdown()
    _initialised_device = None


def lib():
    """The initialised library (initialises on first use)."""
    if _initialised_device is None:
        return init()
    return _lib
