"""ctypes binding of libctd_b200.so (include/ctd_b200.h).  Fails loudly when the library is missing:
there is no fallback implementation of any op."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CTD_B200_LIB") or os.path.join(_HERE, "libctd_b200.so")  # the override is for A/B builds of experiments

_i64, _int, _f32, _f64, _ptr = ctypes.c_int64, ctypes.c_int, ctypes.c_float, ctypes.c_double, ctypes.c_void_p

# name -> argument types (every function returns int unless listed in _RESTYPES)
SIGNATURES = {
    "ctd_set_option": [ctypes.c_char_p, _int],
    "ctd_photometric_fwd_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32, _ptr],
    "ctd_photometric_fwd_f64": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32, _ptr],
    "ctd_photometric_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32, _ptr],
    "ctd_photometric_bwd_f64": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32, _ptr],
    "ctd_photometric_fwd_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32, _ptr],
    "ctd_photometric_fwd_bwd_masked_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32, _ptr],
    "ctd_ssim_fwd_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _f64, _ptr],
    "ctd_ssim_fwd_f64": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _f64, _ptr],
    "ctd_ssim_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _f64, _ptr],
    "ctd_ssim_bwd_f64": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _f64, _ptr],
    "ctd_ssim_fwd_bwd_masked_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _f64, _ptr],
    "ctd_warp_pattern_fwd_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _i64, _ptr],
    "ctd_warp_pattern_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _i64, _ptr],
    "ctd_depth_similarity_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _f32, _f32, _int, _ptr],
    "ctd_disparity_loss_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _f32, _ptr],
    "ctd_xcorrvol_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _ptr],
    "ctd_xcorrvol_f64": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _ptr],
    "ctd_xcorr_disparity_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _ptr],
    "ctd_xcorr_disparity_f64": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _ptr],
    "ctd_sgm_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _f64, _f64, _int, _int, _ptr],
    "ctd_sgm_f64": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _f64, _f64, _int, _int, _ptr],
    "ctd_census_transform_f32": [_ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _ptr],
    "ctd_census_transform_f64": [_ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _ptr],
    "ctd_census_vol_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _int, _ptr],
    "ctd_census_vol_f64": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _int, _ptr],
    "ctd_census_disparity_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _int, _int, _ptr],
    "ctd_census_disparity_f64": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _int, _int, _ptr],
    "ctd_disparity_check_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _int, _ptr],
    "ctd_disparity_check_f64": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _f64, _int, _ptr],
    "ctd_speckle_filter_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _f64, _ptr],
    "ctd_speckle_filter_f64": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _f64, _ptr],
    "ctd_proj_nn_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _ptr],
    "ctd_proj_nn_f64": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _ptr],
    "ctd_nn_f32": [_ptr, _ptr, _ptr, _i64, _i64, _ptr],
    "ctd_nn_f64": [_ptr, _ptr, _ptr, _i64, _i64, _ptr],
    "ctd_crosscheck": [_ptr, _ptr, _ptr, _i64, _i64, _ptr],
    "ctd_lcn_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _f32, _ptr],
    "ctd_lcn_f64": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _f64, _ptr],
    "ctd_pattern_similarity_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _i64, _int, _f32, _ptr],
    "ctd_lcn_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _f32, _ptr],
    "ctd_lcn_cython_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _f32, _ptr],
    "ctd_masked_sums_f32": [_ptr, _ptr, _i64, _ptr, _ptr, _ptr],
    "ctd_host_photometric_fwd_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32],
    "ctd_host_photometric_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32],
    "ctd_host_photometric_fwd_bwd_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32],
    "ctd_host_photometric_fwd_bwd_masked_f32": [_ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _int, _int, _f32],
    "ctd_host_xcorrvol_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _int],
    "ctd_host_proj_nn_f32": [_ptr, _ptr, _ptr, _ptr, _i64, _i64, _i64, _int],
    "ctd_host_nn_f32": [_ptr, _ptr, _ptr, _i64, _i64],
    "ctd_host_crosscheck": [_ptr, _ptr, _ptr, _i64, _i64],
    "ctd_host_lcn_f32": [_ptr, _ptr, _ptr, _i64, _i64, _i64, _int, _f32],
    "ctd_host_begin_batch": [],
    "ctd_host_end_batch": [],
    "ctd_host_end_batch_async": [],
    "ctd_host_wait_batch": [],
}
_RESTYPES = {
    "ctd_last_error": (ctypes.c_char_p, []),
    "ctd_version": (ctypes.c_char_p, []),
    "ctd_launch_count": (ctypes.c_uint64, []),
    "ctd_masked_sums_workspace_bytes": (ctypes.c_int64, []),
    "ctd_host_release": (None, []),
    "ctd_host_batch_stats": (None, [_ptr, _ptr]),
    "ctd_host_graph_stats": (None, [_ptr, _ptr, _ptr]),
}
EXPORTS = sorted(list(SIGNATURES) + list(_RESTYPES))

_lib = None


class CtdError(RuntimeError):
    pass


def lib():
    """The loaded library.  Raises if libctd_b200.so has not been built (python -m
    connecting_the_dots_b200._build, or __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CtdError("libctd_b200.so is not built: run `python -m connecting_the_dots_b200._build` "
                           "(there is no fallback implementation)")
        L = ctypes.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes, fn.restype = args, _int
        for name, (res, args) in _RESTYPES.items():
            fn = getattr(L, name)
            fn.argtypes, fn.restype = args, res
        _lib = L
    return _lib


def call(name, *args):
    """Invoke a status-returning entry point; non-zero status -> CtdError / ValueError-like RuntimeError."""
    L = lib()
    rc = getattr(L, name)(*args)
    if rc != 0:
        raise CtdError("%s failed (%d): %s" % (name, rc, L.ctd_last_error().decode(errors="replace")))


def launch_count():
    return int(lib().ctd_launch_count())


def set_option(name, value):
    call("ctd_set_option", name.encode(), int(value))
