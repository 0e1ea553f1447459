"""ctypes binding of libgrates_b200.so (C ABI declared in include/grates_b200.h).

There is deliberately no fallback: if the shared library is missing (and cannot be built
because nvcc is absent) or no CUDA device is usable, every compute call raises.
"""
import ctypes
import os
import threading

_c_double_p = ctypes.POINTER(ctypes.c_double)
_c_int64_p = ctypes.POINTER(ctypes.c_int64)
_vp = ctypes.c_void_p

GB_OK, GB_ERR_ARGUMENT, GB_ERR_CUDA, GB_ERR_UNSUPPORTED, GB_ERR_MEMORY = 0, 1, 2, 3, 4
GB_VERSION = 203        # must equal GB_VERSION of include/grates_b200.h: the argtypes below describe THAT header

# name -> (restype, argtypes); must list every symbol of include/grates_b200.h
SIGNATURES = {
    "gb_version": (ctypes.c_int, []),
    "gb_last_error": (ctypes.c_char_p, []),
    "gb_device_count": (ctypes.c_int, [ctypes.POINTER(ctypes.c_int)]),
    "gb_trim": (ctypes.c_int, [ctypes.c_int]),
    "gb_plan_create": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp, _vp,
                                      _vp, _vp, ctypes.c_int]),
    "gb_plan_destroy": (ctypes.c_int, [_vp]),
    "gb_plan_info": (ctypes.c_int, [_vp] + [ctypes.POINTER(ctypes.c_int)] * 4),
    "gb_plan_is_symmetric": (ctypes.c_int, [_vp]),
    "gb_plan_is_folded": (ctypes.c_int, [_vp]),
    "gb_synthesis": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp]),
    "gb_synthesis_host": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp]),
    "gb_legendre_table": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp]),
    "gb_plan_set_analysis": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp, _vp]),
    "gb_plan_set_analysis_weights": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp]),
    "gb_analysis": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp]),
    "gb_analysis_host": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp]),
    "gb_synthesis_matrix": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp]),
    "gb_analysis_matrix": (ctypes.c_int, [_vp, _vp, _vp]),
    "gb_covariance_propagation": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp,
                                                 ctypes.c_int, _vp]),
    "gb_covariance_propagation_filtered": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp,
                                                          ctypes.c_int, _vp, _vp, ctypes.c_int, _vp, _vp]),
    "gb_scale_by_degree": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, _vp]),
    "gb_synthesis_weighted": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int, _vp, _vp]),
    "gb_synthesis_orderwise_filtered": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int, _vp, ctypes.c_int, _vp, _vp]),
    "gb_dense_filter_tile_elements": (ctypes.c_int64, [ctypes.c_int64]),
    "gb_dense_filter_prepare": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, ctypes.c_int, _vp]),
    "gb_dense_filter": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, _vp]),
    "gb_orderwise_filter": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, _vp,
                                           ctypes.c_int, _vp]),
    "gb_points_create": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, ctypes.c_int, _vp, _vp, _vp, _vp, _vp,
                                        ctypes.c_int]),
    "gb_points_destroy": (ctypes.c_int, [_vp]),
    "gb_points_synthesis": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp]),
    "gb_points_covariance": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, ctypes.c_int, _vp]),
    "gb_points_adjoint": (ctypes.c_int, [_vp, _vp, ctypes.c_int, _vp, _vp]),
    "gb_points_synthesis_matrix": (ctypes.c_int, [_vp, ctypes.c_int, _vp, _vp]),
    "gb_temporal_rms": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int64, _vp, ctypes.c_int, _vp]),
    "gb_weighted_moments": (ctypes.c_int, [_vp, _vp, _vp, ctypes.c_int, ctypes.c_int64, _vp, ctypes.c_int, _vp]),
    "gb_ravel_coefficients": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, _vp]),
    "gb_quadratic_forms": (ctypes.c_int, [_vp, ctypes.c_int64, _vp, ctypes.c_int, _vp, ctypes.c_int, _vp]),
    "gb_gradient_coefficients": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int, _vp]),
    "gb_rotate_to_local": (ctypes.c_int, [_vp, _vp, ctypes.c_int, ctypes.c_int64, ctypes.c_int, _vp]),
    "gb_host_alloc":(ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_uint64]),
    "gb_host_free": (ctypes.c_int, [_vp]),
    "gb_probe_fp64_peak": (ctypes.c_int, [ctypes.c_int, _c_double_p, _c_double_p]),
    "gb_plan_set_profiling": (ctypes.c_int, [_vp, ctypes.c_int]),
    "gb_plan_stage_times": (ctypes.c_int, [_vp, _c_double_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]),
    "gb_launch_count": (ctypes.c_int64, [ctypes.c_int]),
    "gb_dgemm": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_double,
                                _vp, ctypes.c_int64, _vp, ctypes.c_int64, ctypes.c_double, _vp, ctypes.c_int64, ctypes.c_int,
                                ctypes.c_int, _vp]),
    "gb_dpotrf_upper": (ctypes.c_int, [_vp, ctypes.c_int64, ctypes.c_int64, _vp, ctypes.c_int, _vp]),
    "gb_dtrsm_upper": (ctypes.c_int, [ctypes.c_int, _vp, ctypes.c_int64, ctypes.c_int64, _vp, ctypes.c_int64, ctypes.c_int64,
                                      ctypes.c_int, _vp]),
}

_lock = threading.Lock()
_lib = None


def library_path():
    # GRATES_B200_LIBRARY: a development build of the same ABI (e.g. one compiled with -DGB_TRACE)
    return os.environ.get("GRATES_B200_LIBRARY") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib",
                                                                 "libgrates_b200.so")


def load():
    """Load and return the CDLL.  The library is rebuilt first when it is missing, older than its sources or the
    header, or when GRATES_B200_REBUILD is set; a current library loads without nvcc (the GPU box has the prebuilt
    file).  A library of another ABI version is refused rather than called with the wrong argument types."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        path = library_path()
        from . import build as _build
        if os.environ.get("GRATES_B200_REBUILD") or _build.needs_build():
            try:
                _build.build(force=True)
            except RuntimeError:
                if not os.path.exists(path):
                    raise
                import warnings
                warnings.warn("libgrates_b200.so is older than its sources and could not be rebuilt (no nvcc?)")
        if not os.path.exists(path):
            raise RuntimeError("libgrates_b200.so is missing (%s); run `python -m grates_b200.build`. "
                               "grates_b200 has no CPU fallback." % path)
        lib = ctypes.CDLL(path)
        lib.gb_version.restype = ctypes.c_int
        if lib.gb_version() != GB_VERSION:
            raise RuntimeError("libgrates_b200.so has ABI version %d, this package expects %d; rebuild it with "
                               "`python -m grates_b200.build`" % (lib.gb_version(), GB_VERSION))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError here means header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def check(rc):
    """Turn a C ABI return code into the Python exception the reference would raise."""
    if rc == GB_OK:
        return
    msg = load().gb_last_error().decode("utf-8", "replace")
    if rc == GB_ERR_ARGUMENT:
        raise ValueError(msg)
    if rc == GB_ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == GB_ERR_MEMORY:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def device_count():
    n = ctypes.c_int(0)
    check(load().gb_device_count(ctypes.byref(n)))
    return n.value


def require_device():
    """Fail loudly when there is nothing to run on (no silent CPU path)."""
    try:
        n = device_count()
    except RuntimeError as exc:
        raise RuntimeError("grates_b200 needs a CUDA device (B200, sm_100a): %s" % exc) from None
    if n < 1:
        raise RuntimeError("grates_b200 needs a CUDA device (B200, sm_100a); none is visible")
    return n
