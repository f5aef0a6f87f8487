"""ctypes binding of the C ABI declared in include/hrb.h (hopperrender_b200/libhrb.so).

There is deliberately no fallback: if the CUDA library is missing or fails to load, importing the
product raises.  The CPU oracle under oracle/ is test infrastructure and is never imported here.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhrb.so")


class hrb_ofc_desc(C.Structure):
    _fields_ = [
        ("frame_height", C.c_int), ("frame_width", C.c_int), ("input_stride", C.c_int), ("output_stride", C.c_int),
        ("delta_scalar", C.c_int), ("neighbor_scalar", C.c_int), ("black_level", C.c_float), ("white_level", C.c_float),
        ("max_calc_res", C.c_int), ("is_hdr", C.c_int), ("device_ordinal", C.c_int), ("cuda_stream", C.c_void_p),
    ]


class hrb_ofc_state(C.Structure):
    _fields_ = [
        ("frame_width", C.c_int), ("frame_height", C.c_int), ("input_stride", C.c_int), ("output_stride", C.c_int),
        ("output_black_level", C.c_float), ("output_white_level", C.c_float),
        ("res_scalar", C.c_int), ("flow_width", C.c_int), ("flow_height", C.c_int), ("search_radius", C.c_int),
        ("ofc_calc_time", C.c_double), ("ofc_avg_calc_time", C.c_double), ("ofc_peak_calc_time", C.c_double),
        ("ofc_calc_count", C.c_int), ("ofc_calc_time_sum", C.c_double), ("warp_calc_time", C.c_double),
        ("delta_scalar", C.c_int), ("neighbor_bias_scalar", C.c_int),
        ("total_frame_delta", C.c_uint), ("frame_count", C.c_uint),
    ]


class hrb_ofc_params(C.Structure):
    _fields_ = [("search_radius", C.c_int), ("delta_scalar", C.c_int), ("neighbor_bias_scalar", C.c_int),
                ("black_level", C.c_float), ("white_level", C.c_float)]


class hrb_ofc_profile(C.Structure):
    _fields_ = [("ms_ingest", C.c_double), ("ms_search", C.c_double), ("ms_blur", C.c_double), ("ms_warp", C.c_double),
                ("ms_copy", C.c_double), ("n_ingest", C.c_uint64), ("n_search", C.c_uint64), ("n_blur", C.c_uint64),
                ("n_warp", C.c_uint64), ("n_copy", C.c_uint64)]


class hrb_frame_planes(C.Structure):
    _fields_ = [("y", C.c_void_p), ("y_pitch_bytes", C.c_size_t), ("uv", C.c_void_p), ("uv_pitch_bytes", C.c_size_t)]


class hrb_delivery_desc(C.Structure):
    _fields_ = [("source_frame_time", C.c_longlong), ("target_frame_time", C.c_longlong), ("frame_output_mode", C.c_int),
                ("scene_change_threshold", C.c_int), ("active", C.c_int), ("auto_adjust", C.c_int)]


class hrb_delivery_frame(C.Structure):
    _fields_ = [("source", C.c_uint), ("index", C.c_int), ("blend", C.c_double), ("step", C.c_ulonglong)]


class hrb_delivery_outcome(C.Structure):
    _fields_ = [("warped", C.c_int), ("scene_change", C.c_int), ("delta1", C.c_longlong), ("delta2", C.c_longlong),
                ("frame_delta", C.c_uint)]


class hrb_side_data(C.Structure):
    _fields_ = [("guid", C.c_uint8 * 16), ("data", C.c_void_p), ("bytes", C.c_size_t)]


# name -> (restype, argtypes); every symbol include/hrb.h declares
_P = C.c_void_p
PROTOTYPES = {
    "hrb_ofc_create": (C.c_int, [C.POINTER(_P), C.POINTER(hrb_ofc_desc)]),
    "hrb_ofc_destroy": (None, [_P]),
    "hrb_ofc_update_frame": (C.c_int, [_P, _P]),
    "hrb_ofc_calculate_optical_flow": (C.c_int, [_P]),
    "hrb_ofc_warp_frames": (C.c_int, [_P, C.c_float, C.c_int]),
    "hrb_ofc_warp_frames_batch": (C.c_int, [_P, C.c_int, C.POINTER(C.c_float), C.c_int]),
    "hrb_ofc_copy_frame": (C.c_int, [_P]),
    "hrb_ofc_download_frame": (C.c_int, [_P, _P]),
    "hrb_ofc_get_state": (C.c_int, [_P, C.POINTER(hrb_ofc_state)]),
    "hrb_ofc_peek_state": (C.c_int, [_P, C.POINTER(hrb_ofc_state)]),
    "hrb_ofc_set_params": (C.c_int, [_P, C.POINTER(hrb_ofc_params)]),
    "hrb_ofc_set_frame_count": (C.c_int, [_P, C.c_uint]),
    "hrb_ofc_reset": (C.c_int, [_P]),
    "hrb_ofc_update_frame_device": (C.c_int, [_P, _P]),
    "hrb_ofc_output_device_ptr": (C.c_int, [_P, C.POINTER(_P)]),
    "hrb_ofc_update_frame_async": (C.c_int, [_P, _P]),
    "hrb_ofc_wait_upload": (C.c_int, [_P]),
    "hrb_ofc_download_frame_async": (C.c_int, [_P, _P, C.POINTER(C.c_ulonglong)]),
    "hrb_ofc_wait_download": (C.c_int, [_P, C.c_ulonglong]),
    "hrb_ofc_calculate_optical_flow_async": (C.c_int, [_P]),
    "hrb_ofc_synchronize": (C.c_int, [_P]),
    "hrb_ofc_stream": (C.c_int, [_P, C.POINTER(_P)]),
    "hrb_ofc_update_frame_planes": (C.c_int, [_P, C.POINTER(hrb_frame_planes)]),
    "hrb_ofc_warp_frames_to": (C.c_int, [_P, C.c_int, C.POINTER(C.c_float), C.c_int, C.POINTER(hrb_frame_planes)]),
    "hrb_ofc_copy_frame_to": (C.c_int, [_P, C.POINTER(hrb_frame_planes)]),
    "hrb_host_register": (C.c_int, [_P, C.c_size_t]),
    "hrb_host_unregister": (C.c_int, [_P]),
    "hrb_host_alloc": (C.c_int, [C.POINTER(_P), C.c_size_t]),
    "hrb_host_free": (C.c_int, [_P]),
    "hrb_delivery_create": (C.c_int, [C.POINTER(_P), _P, C.POINTER(hrb_delivery_desc)]),
    "hrb_delivery_destroy": (None, [_P]),
    "hrb_delivery_next_count": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "hrb_delivery_step": (C.c_int, [_P, C.POINTER(hrb_delivery_frame), C.c_int, C.POINTER(C.c_int)]),
    "hrb_delivery_step_to": (C.c_int, [_P, C.POINTER(hrb_frame_planes), C.c_int, C.POINTER(hrb_delivery_frame), C.POINTER(C.c_int)]),
    "hrb_delivery_outcome_of": (C.c_int, [_P, C.c_ulonglong, C.c_int, C.POINTER(hrb_delivery_outcome)]),
    "hrb_delivery_set": (C.c_int, [_P, C.POINTER(hrb_delivery_desc)]),
    "hrb_delivery_new_segment": (C.c_int, [_P, C.c_double]),
    "hrb_ofc_set_output_stripe": (C.c_int, [_P, C.c_int, C.c_int]),
    "hrb_split_plan": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "hrb_split_create": (C.c_int, [C.POINTER(_P), C.POINTER(_P), C.c_int]),
    "hrb_split_destroy": (None, [_P]),
    "hrb_split_stripe": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "hrb_split_calculate_optical_flow": (C.c_int, [_P]),
    "hrb_split_calculate_optical_flow_async": (C.c_int, [_P]),
    "hrb_flow_batch_create": (C.c_int, [C.POINTER(_P), C.POINTER(_P), C.c_int]),
    "hrb_flow_batch_destroy": (None, [_P]),
    "hrb_flow_batch_calculate_optical_flow": (C.c_int, [_P]),
    "hrb_flow_batch_calculate_optical_flow_async": (C.c_int, [_P]),
    "hrb_ofc_set_tap_mode": (C.c_int, [_P, C.c_int]),
    "hrb_ofc_num_passes": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "hrb_ofc_pass_info": (C.c_int, [_P, C.c_int] + [C.POINTER(C.c_int)] * 5),
    "hrb_ofc_read_pass_tap": (C.c_int, [_P, C.c_int, C.c_int, _P, C.c_size_t]),
    "hrb_ofc_read_buffer": (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    "hrb_ofc_write_flow": (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    "hrb_ofc_set_profile": (C.c_int, [_P, C.c_int]),
    "hrb_ofc_profile_read": (C.c_int, [_P, C.POINTER(hrb_ofc_profile)]),
    "hrb_ofc_profile_reset": (C.c_int, [_P]),
    "hrb_ofc_set_search_variant": (C.c_int, [_P, C.c_int]),
    "hrb_ofc_set_flow_overlap": (C.c_int, [_P, C.c_int]),
    "hrb_ofc_join_flow": (C.c_int, [_P]),
    "hrb_ofc_set_side_data": (C.c_int, [_P, C.POINTER(hrb_side_data), C.c_int]),
    "hrb_ofc_get_side_data": (C.c_int, [_P, C.POINTER(hrb_side_data), C.c_int, C.POINTER(C.c_int)]),
    "hrb_ofc_debug_timeline": (C.c_int, [_P, C.c_size_t]),
    "hrb_ofc_debug_timeline_read": (C.c_int, [_P, C.c_void_p, C.c_size_t]),
    "hrb_kernel_launch_count": (C.c_uint64, []),
    "hrb_microbench_sad_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "hrb_last_error": (C.c_char_p, []),
    "hrb_version": (C.c_char_p, []),
}

HRB_OK, HRB_ERR_INVALID_ARG, HRB_ERR_CUDA, HRB_ERR_BLEND_RANGE, HRB_ERR_NO_DEVICE, HRB_ERR_STATE = range(6)
TAP_WINDOW_SUMS, TAP_WINDOW_LAYER, TAP_OFFSETS = 0, 1, 2
DELIVERY_MAX_FRAMES = 16
BUF_OFFSET_ARRAY, BUF_FLOW_FOR_WARP, BUF_FLOW_LATEST, BUF_OUTPUT_FRAME, BUF_RAW_FRAME_DELTA, BUF_FLOW_PEAK = range(6)

_lib = None


def load():
    """Load libhrb.so once and attach the prototypes.  Raises if the library is absent (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C hopperrender_b200/csrc`. hopperrender_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_LOCAL)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().hrb_last_error().decode("utf-8", "replace")
