"""ctypes binding of include/ctcx.h. There is no CPU fallback: if the CUDA library is missing and
cannot be built, or no CUDA device is present, the op raises."""
import ctypes
import os

from . import build as _build

_i64p = ctypes.POINTER(ctypes.c_int64)
_i64pp = ctypes.POINTER(_i64p)
_vp = ctypes.c_void_p


class CtcxSizes(ctypes.Structure):
    _fields_ = [("n_decoded", _i64p), ("max_decoded", _i64p), ("n_alignment", _i64p),
                ("max_alignment", _i64p)]


class CtcxLimits(ctypes.Structure):
    _fields_ = [("max_beam_width", ctypes.c_int), ("max_classes", ctypes.c_int),
                ("max_top_paths", ctypes.c_int)]


class CtcxHostResult(ctypes.Structure):
    _fields_ = [("top_paths", ctypes.c_int), ("n_decoded", _i64p), ("n_alignment", _i64p),
                ("decoded_indices", _i64pp), ("decoded_values", _i64pp), ("decoded_shape", _i64pp),
                ("alignment_indices", _i64pp), ("alignment_values", _i64pp),
                ("alignment_shape", _i64pp), ("log_probability", ctypes.POINTER(ctypes.c_float)),
                ("flags", ctypes.c_int32), ("log_probability_f64", ctypes.POINTER(ctypes.c_double))]


# every symbol include/ctcx.h declares (tests check that the library exports exactly these)
EXPORTS = ("ctcx_strerror", "ctcx_last_cuda_error", "ctcx_error_batch_index", "ctcx_get_limits",
           "ctcx_workspace_bytes", "ctcx_decode_f32", "ctcx_decode_f64", "ctcx_decode_scorer_f32",
           "ctcx_decode_half", "ctcx_decode_view", "ctcx_hostin_staging_bytes", "ctcx_decode_hostin",
           "ctcx_pack_f32", "ctcx_pack_f64", "ctcx_pack_compact", "ctcx_finish", "ctcx_result_bytes", "ctcx_result_copy_async", "ctcx_result_parse", "ctcx_decode_host_f32", "ctcx_decode_host_f64", "ctcx_free_host",
           "ctcx_stream_workspace_bytes", "ctcx_stream_reset", "ctcx_stream_step_f32", "ctcx_stream_top_paths",
           "ctcx_stream_workspace_bytes_v", "ctcx_stream_reset_v", "ctcx_stream_step_v",
           # measurement and test hooks
           "ctcx_workspace_views", "ctcx_profile_enable", "ctcx_profile_get", "ctcx_debug_set_cycles_buffer",
           "ctcx_debug_set_beam_impl", "ctcx_debug_math_f32", "ctcx_debug_math_f64", "ctcx_debug_prepass")

F32, F16, BF16, F64 = 0, 1, 2, 3  # CTCX_F32 ... (include/ctcx.h)

_lib = None


def load():
    """Load (building first if the sources are newer) lib/libctcx.so. Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if _build.is_stale():
        try:
            _build.build()
        except Exception as e:  # no nvcc on this box and no library built from these sources
            # never load a library built from OTHER sources silently: bit-exactness is the contract
            raise RuntimeError(
                "ctcx: the CUDA library %s is %s and could not be (re)built (%s). "
                "There is no CPU fallback." % (path, "stale" if os.path.exists(path) else "missing", e))
    lib = ctypes.CDLL(path)
    lib.ctcx_strerror.restype = ctypes.c_char_p
    lib.ctcx_strerror.argtypes = [ctypes.c_int]
    lib.ctcx_last_cuda_error.restype = ctypes.c_char_p
    lib.ctcx_get_limits.argtypes = [ctypes.POINTER(CtcxLimits)]
    lib.ctcx_workspace_bytes.restype = ctypes.c_size_t
    lib.ctcx_workspace_bytes.argtypes = [ctypes.c_int] * 5
    lib.ctcx_decode_f32.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int,
                                    ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp,
                                    ctypes.c_size_t, _vp, ctypes.POINTER(CtcxSizes),
                                    ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_decode_f64.argtypes = lib.ctcx_decode_f32.argtypes
    lib.ctcx_decode_scorer_f32.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, ctypes.c_int,
                                           ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp, _vp,
                                           ctypes.c_size_t, _vp, ctypes.POINTER(CtcxSizes),
                                           ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_decode_half.argtypes = [_vp, ctypes.c_int, _vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp,
                                     ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     _vp, ctypes.c_size_t, _vp, ctypes.POINTER(CtcxSizes),
                                     ctypes.POINTER(ctypes.c_int32)]
    _i = ctypes.c_int
    lib.ctcx_error_batch_index.argtypes = []
    lib.ctcx_decode_view.argtypes = [_vp, _i, ctypes.c_int64, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp,
                                     ctypes.c_size_t, _vp, ctypes.POINTER(CtcxSizes),
                                     ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_hostin_staging_bytes.restype = ctypes.c_size_t
    lib.ctcx_hostin_staging_bytes.argtypes = [_i] * 4
    lib.ctcx_decode_hostin.argtypes = [_vp, _i, ctypes.c_int64, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _vp,
                                       ctypes.c_size_t, _vp, ctypes.c_size_t, _vp, _vp,
                                       ctypes.POINTER(CtcxSizes), ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_debug_set_beam_impl.argtypes = [_i]
    lib.ctcx_debug_set_beam_impl.restype = None
    lib.ctcx_pack_f32.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [_vp] * 6 + [_vp, _vp]
    lib.ctcx_pack_f64.argtypes = lib.ctcx_pack_f32.argtypes
    lib.ctcx_pack_compact.argtypes = [_vp, _i, _i, _i, _i, _vp, ctypes.c_size_t, _vp]
    lib.ctcx_finish.argtypes = [_vp, _i, _i, _i, _vp, ctypes.POINTER(CtcxSizes), ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_result_bytes.restype = ctypes.c_size_t
    lib.ctcx_result_bytes.argtypes = [_i]
    lib.ctcx_result_copy_async.argtypes = [_vp, _i, _i, _i, _vp, ctypes.c_size_t, _vp]
    lib.ctcx_result_parse.argtypes = [_vp, _i, _i, _i, ctypes.POINTER(CtcxSizes), ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_decode_host_f32.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _vp,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int,
                                         ctypes.POINTER(ctypes.POINTER(CtcxHostResult))]
    lib.ctcx_decode_host_f64.argtypes = lib.ctcx_decode_host_f32.argtypes
    lib.ctcx_free_host.argtypes = [ctypes.POINTER(CtcxHostResult)]
    lib.ctcx_free_host.restype = None
    lib.ctcx_workspace_views.argtypes = [_vp, ctypes.c_int, ctypes.c_int, ctypes.c_int] + [_vp] * 5
    lib.ctcx_stream_workspace_bytes.restype = ctypes.c_size_t
    lib.ctcx_stream_workspace_bytes.argtypes = [ctypes.c_int] * 5
    lib.ctcx_stream_reset.argtypes = [_vp, ctypes.c_size_t] + [ctypes.c_int] * 5 + [_vp]
    lib.ctcx_stream_step_f32.argtypes = [_vp] + [ctypes.c_int] * 5 + [_vp, ctypes.c_int, _vp, ctypes.c_int, _vp]
    lib.ctcx_stream_workspace_bytes_v.restype = ctypes.c_size_t
    lib.ctcx_stream_workspace_bytes_v.argtypes = [ctypes.c_int] * 6
    lib.ctcx_stream_reset_v.argtypes = [_vp, ctypes.c_size_t] + [ctypes.c_int] * 6 + [_vp]
    lib.ctcx_stream_step_v.argtypes = [_vp, ctypes.c_size_t] + [_i] * 5 + [_vp, _i, ctypes.c_int64, _i, _vp, _i,
                                                                            _vp, _vp]
    lib.ctcx_stream_top_paths.argtypes = [_vp] + [ctypes.c_int] * 5 + [ctypes.c_int, ctypes.c_int, _vp,
                                                                      ctypes.POINTER(CtcxSizes),
                                                                      ctypes.POINTER(ctypes.c_int32)]
    lib.ctcx_profile_enable.argtypes = [ctypes.c_int]
    lib.ctcx_profile_enable.restype = None
    lib.ctcx_profile_get.argtypes = [ctypes.POINTER(ctypes.c_float)]
    lib.ctcx_profile_get.restype = None
    lib.ctcx_debug_set_cycles_buffer.argtypes = [_vp]
    lib.ctcx_debug_set_cycles_buffer.restype = None
    lib.ctcx_debug_math_f32.argtypes = [ctypes.c_int, _vp, _vp, ctypes.c_int, _vp]
    lib.ctcx_debug_math_f64.argtypes = [ctypes.c_int, _vp, _vp, ctypes.c_int, _vp]
    lib.ctcx_debug_prepass.argtypes = [_i, _vp, _i, _i, _i, _i, ctypes.c_longlong, _i, _i, _vp, _vp, _vp,
                                       ctypes.POINTER(_i), _vp]
    _lib = lib
    return lib
