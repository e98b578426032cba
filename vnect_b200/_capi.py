"""ctypes binding of libvnect_b200.so (C ABI declared in include/vnect_b200.h).

There is no CPU fallback: if the CUDA library is missing the import of this module's users fails loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libvnect_b200.so")

OK, E_INVALID, E_CUDA, E_WEIGHT, E_ZERO_DT, E_UNSUPPORTED, E_NUMERIC = 0, -1, -2, -3, -4, -5, -6
MAX_SCALES = 4
STREAM_STATE_DOUBLES = 7 * 21 * 5 + 6


class Config(C.Structure):
    _fields_ = [
        ("device", C.c_int32),
        ("box_size", C.c_int32),
        ("n_scales", C.c_int32),
        ("scales", C.c_double * MAX_SCALES),
        ("max_frames", C.c_int32),
        ("max_streams", C.c_int32),
        ("max_input_h", C.c_int32),
        ("max_input_w", C.c_int32),
        ("filters", C.c_int32),
    ]


FMT_BGR, FMT_NV12, FMT_I420 = 0, 1, 2


class YuvLayout(C.Structure):
    """vnect_yuv_layout: where the planes of each YUV 4:2:0 frame are (bytes, relative to the frame's start)."""
    _fields_ = [
        ("format", C.c_int32),
        ("reserved", C.c_int32),
        ("y_pitch", C.c_int64),
        ("uv_pitch", C.c_int64),
        ("u_offset", C.c_int64),
        ("v_offset", C.c_int64),
        ("frame_stride", C.c_int64),
    ]


class Frame(C.Structure):
    """vnect_frame: one frame of a mixed-size batch -- its address, full size, row pitch and (YUV) chroma layout."""
    _fields_ = [
        ("data", C.c_void_p),
        ("height", C.c_int32),
        ("width", C.c_int32),
        ("pitch", C.c_int64),
        ("uv_pitch", C.c_int64),
        ("u_offset", C.c_int64),
        ("v_offset", C.c_int64),
    ]


# every symbol include/vnect_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_YL = C.POINTER(YuvLayout)
_FR = C.POINTER(Frame)
SIGNATURES = {
    "vnect_create": (C.c_int, [C.POINTER(_P), C.POINTER(Config)]),
    "vnect_set_weight": (C.c_int, [_P, C.c_char_p, _P, C.POINTER(C.c_int64), C.c_int32]),
    "vnect_crc32c": (C.c_uint32, [_P, C.c_uint64]),
    "vnect_finalize": (C.c_int, [_P]),
    "vnect_forward": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P]),
    "vnect_estimate": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "vnect_submit": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "vnect_wait": (C.c_int, [_P, C.c_int32]),
    "vnect_track_set_box": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "vnect_track_get_box": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    "vnect_track": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P, _P, _P, _P]),
    "vnect_estimate_device": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P, _P, _P]),
    "vnect_submit_yuv": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, _YL, _P, _P, _P, _P, _P]),
    "vnect_estimate_device_yuv": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _YL, _P, _P, _P, _P, _P]),
    "vnect_track_yuv": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, _YL, _P, _P, _P, _P, _P, _P]),
    "vnect_submit_frames": (C.c_int, [_P, C.c_int32, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "vnect_estimate_device_frames": (C.c_int, [_P, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "vnect_track_frames": (C.c_int, [_P, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "vnect_submit_track_frames": (C.c_int, [_P, C.c_int32, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "vnect_track_device_frames": (C.c_int, [_P, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "vnect_track_set_boxes": (C.c_int, [_P, C.c_int32, _P, _P]),
    "vnect_set_orientations": (C.c_int, [_P, C.c_int32, _P, _P]),
    "vnect_get_orientation": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    "vnect_request_scores": (C.c_int, [_P, _P]),
    "vnect_set_track_recovery": (C.c_int, [_P, C.c_int32, _P, _P]),
    "vnect_get_track_recovery": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_double)]),
    "vnect_submit_sequence": (C.c_int, [_P, C.c_int32, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "vnect_estimate_device_sequence": (C.c_int, [_P, _FR, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "vnect_postprocess_sequence": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, _P, _P, _P, C.c_double, C.c_int32,
                                             C.c_int32, _P, _P, _P]),
    "vnect_preprocess": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _P, _P]),
    "vnect_postprocess": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, _P, _P, _P, C.c_double, C.c_int32, C.c_int32, _P, _P, _P]),
    "vnect_track_postprocess": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "vnect_filter": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_double, _P]),
    "vnect_export_stream_state": (C.c_int, [_P, C.c_int32, _P]),
    "vnect_import_stream_state": (C.c_int, [_P, C.c_int32, _P]),
    "vnect_get_raw_argmax": (C.c_int, [_P, C.c_int32, _P]),
    "vnect_joints2angles": (C.c_int, [_P, _P, C.c_int32, _P, _P, _P]),
    "vnect_reset_stream": (C.c_int, [_P, C.c_int32]),
    "vnect_set_stream": (C.c_int, [_P, _P]),
    "vnect_set_packed_results": (C.c_int, [_P, _P]),
    "vnect_synchronize": (C.c_int, [_P]),
    "vnect_get_tap": (C.c_int, [_P, C.c_char_p, C.c_int32, _P, C.c_int64, C.POINTER(C.c_int32)]),
    "vnect_get_input": (C.c_int, [_P, C.c_int32, _P, C.c_int64, C.POINTER(C.c_int32)]),
    "vnect_get_maps": (C.c_int, [_P, C.c_int32, _P, C.c_int64, C.POINTER(C.c_int32)]),
    "vnect_check_finite": (C.c_int, [_P, C.c_int32, _P]),
    "vnect_launch_count": (C.c_int64, [_P]),
    "vnect_info": (C.c_double, [_P, C.c_char_p]),
    "vnect_time_forward": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_float), _P]),
    "vnect_time_prepost": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "vnect_step_name": (C.c_char_p, [_P, C.c_int32]),
    "vnect_step_path": (C.c_int, [_P, C.c_int32, C.POINTER(C.c_int32)]),
    "vnect_last_error": (C.c_char_p, [_P]),
    "vnect_version": (C.c_char_p, []),
    "vnect_destroy": (None, [_P]),
}

_lib = None


def load_library():
    """dlopen the in-tree CUDA library; raises if it has not been built (python __graft_entry__.py build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: vnect_b200 has no CPU path. Build it with `make -C vnect_b200/csrc` "
            "(or `python -c 'import __graft_entry__ as g; g.build()'`).")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def raise_for(lib, handle, code):
    if code == OK:
        return
    msg = lib.vnect_last_error(handle)
    msg = msg.decode() if msg else f"vnect error {code}"
    if code == E_ZERO_DT:
        raise ZeroDivisionError(msg)  # what the reference's OneEuroFilter raises (src/OneEuroFilter.py:66)
    if code == E_INVALID:
        raise ValueError(msg)
    if code == E_WEIGHT:
        raise KeyError(msg)
    if code == E_UNSUPPORTED:
        raise NotImplementedError(msg)
    if code == E_NUMERIC:
        raise FloatingPointError(msg)
    raise RuntimeError(msg)
