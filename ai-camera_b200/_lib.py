"""ctypes binding of ``libaicam.so`` (the C ABI declared in ``include/aicam.h``).

There is no CPU fallback: if the library is missing or a call fails, an exception is
raised.  Device memory, streams and host pinned buffers come from PyTorch (plumbing);
every kernel is in the library.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libaicam.so")

OK = 0
KIND_YOLOV8, KIND_REID = 1, 2


class AicamError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("aicam error %d: %s" % (code, message))
        self.code = code


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("batch", "h", "w", "cin", "cout", "ksize", "stride", "act",
                                       "res_mode", "out_f32")]


class ChainStage(C.Structure):
    _fields_ = [("cin", C.c_int), ("cout", C.c_int), ("ksize", C.c_int), ("act", C.c_int), ("nsrc", C.c_int),
                ("src_buf", C.c_int * 2), ("src_coff", C.c_int * 2), ("src_c", C.c_int * 2),
                ("res_buf", C.c_int), ("res_coff", C.c_int), ("res_mode", C.c_int)]


class ChainDesc(C.Structure):
    _fields_ = [("batch", C.c_int), ("h", C.c_int), ("w", C.c_int), ("in_c", C.c_int), ("nstages", C.c_int),
                ("st", ChainStage * 5), ("out_f32", C.c_int)]


class Letterbox(C.Structure):
    _fields_ = [("ratio", C.c_double), ("pad_w", C.c_double), ("pad_h", C.c_double)]


class NmsParams(C.Structure):
    _fields_ = [("score_thr", C.c_float), ("iou_thr", C.c_float), ("topk", C.c_int),
                ("max_candidates", C.c_int), ("frame_h", C.c_int), ("frame_w", C.c_int)]


class FrameDesc(C.Structure):
    _fields_ = [("data", C.c_void_p), ("chroma", C.c_void_p), ("h", C.c_int), ("w", C.c_int), ("pitch", C.c_int),
                ("kind", C.c_int)]


class StreamFilter(C.Structure):
    _fields_ = [("score_thr", C.c_float), ("iou_thr", C.c_float), ("min_confidence", C.c_float), ("reserved", C.c_int),
                ("class_mask_lo", C.c_uint64), ("class_mask_hi", C.c_uint64)]


class StreamAssoc(C.Structure):
    _fields_ = [("max_cosine_distance", C.c_double), ("max_iou_distance", C.c_double), ("max_age", C.c_int),
                ("n_init", C.c_int)]


class TrackerConfig(C.Structure):
    _fields_ = [("n_streams", C.c_int), ("max_tracks", C.c_int), ("max_dets", C.c_int),
                ("feature_dim", C.c_int), ("max_cosine_distance", C.c_double),
                ("max_iou_distance", C.c_double), ("max_age", C.c_int), ("n_init", C.c_int),
                ("nn_budget", C.c_int), ("device", C.c_int)]


class OverlayItem(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("type", "x1", "y1", "x2", "y2", "color", "slot", "reserved")]


class TensorInfo(C.Structure):
    _fields_ = [("name", C.c_char * 32), ("dtype", C.c_int), ("ndim", C.c_int), ("shape", C.c_int * 4),
                ("is_dynamic", C.c_int)]


_P = C.c_void_p
_I = C.c_int
# name -> (restype, argtypes); every symbol include/aicam.h declares
SIGNATURES = {
    "aicam_version": (_I, []),
    "aicam_last_error": (C.c_char_p, []),
    "aicam_launch_count": (C.c_uint64, []),
    "aicam_profile_enable": (_I, [_I]),
    "aicam_profile_conv": (_I, [C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "aicam_debug_timeline": (_I, [_I, C.POINTER(C.c_longlong), _I]),
    "aicam_engine_create": (_I, [C.c_char_p, _I, _I, C.POINTER(_P)]),
    "aicam_engine_destroy": (None, [_P]),
    "aicam_engine_kind": (_I, [_P]),
    "aicam_engine_max_batch": (_I, [_P]),
    "aicam_engine_num_classes": (_I, [_P]),
    "aicam_engine_num_anchors": (_I, [_P]),
    "aicam_engine_flops_per_item": (C.c_double, [_P]),
    "aicam_engine_num_launches": (_I, [_P]),
    "aicam_engine_io_count": (_I, [_P, _I]),
    "aicam_engine_io_info": (_I, [_P, _I, _I, _I, C.POINTER(TensorInfo)]),
    "aicam_engine_set_bias": (_I, [_P, C.c_char_p, _P, _I]),
    "aicam_engine_get_bias": (_I, [_P, C.c_char_p, _P, _I]),
    "aicam_yolo_forward": (_I, [_P, _P, _I, _P, _P]),
    "aicam_yolo_forward_s2d": (_I, [_P, _P, _I, _P, _P]),
    "aicam_engine_accepts_s2d": (_I, [_P]),
    "aicam_yolo_detect": (_I, [_P, _P, _I, _I, C.POINTER(NmsParams), _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "aicam_engine_fused_decode": (_I, [_P]),
    "aicam_reid_forward": (_I, [_P, _P, _I, _P, _P, _P]),
    "aicam_reid_forward_nhwc8": (_I, [_P, _P, _I, _P, _P, _P]),
    "aicam_engine_accepts_nhwc8": (_I, [_P]),
    "aicam_nchw_to_nhwc4": (_I, [_P, _I, _I, _I, _P, _P]),
    "aicam_conv2d": (_I, [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _P]),
    "aicam_conv2d_padded": (_I, [C.POINTER(ConvDesc), _P, _P, _P, _P, _P, _I, _I, _P]),
    "aicam_conv_chain": (_I, [C.POINTER(ChainDesc), _P, C.POINTER(_P), C.POINTER(_P), _P, _P]),
    "aicam_conv_chain_bench": (_I, [C.POINTER(ChainDesc), _I, C.POINTER(C.c_double), _P]),
    "aicam_conv2d_bench": (_I, [C.POINTER(ConvDesc), _I, C.POINTER(C.c_double), _P]),
    "aicam_reid_stem_pool": (_I, [_P, _I, _I, _I, _P, _P, _P, _P]),
    "aicam_letterbox_params": (_I, [_I, _I, C.POINTER(Letterbox)]),
    "aicam_preprocess": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "aicam_preprocess_nv12": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "aicam_nv12_to_bgr": (_I, [_P, _I, _I, _I, _P, _P]),
    "aicam_frame_table_create": (_I, [_I, _I, _I, _I, C.POINTER(_P)]),
    "aicam_frame_table_destroy": (None, [_P]),
    "aicam_frame_table_set": (_I, [_P, C.POINTER(FrameDesc), _I, _P]),
    "aicam_frame_table_set_present": (_I, [_P, C.POINTER(FrameDesc), _P, _I, _P]),
    "aicam_frame_table_present": (_P, [_P]),
    "aicam_frame_table_set_filters": (_I, [_P, C.POINTER(StreamFilter), _I]),
    "aicam_preprocess_table": (_I, [_P, _I, _P, _P]),
    "aicam_yolo_detect_table": (_I, [_P, _P, _I, _P, C.POINTER(NmsParams), _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    "aicam_reid_crops_table": (_I, [_P, _P, _P, _P, _P, _I, C.c_float, C.c_uint64, C.c_uint64, _I, _I, _P, _P, _P, _P,
                                    _P, _P, _P]),
    "aicam_decode_nms": (_I, [_P, _I, _I, _I, C.POINTER(NmsParams), _P, _P, _P, _P, _P, _P,
                              C.c_size_t, _P]),
    "aicam_decode_nms_workspace": (C.c_size_t, [_I, _I, C.POINTER(NmsParams)]),
    "aicam_decode": (_I, [_P, _I, _I, _I, _P, _P, _P, _P]),
    "aicam_nms": (_I, [_P, _P, _P, _I, _I, C.POINTER(NmsParams), _P, _P, _P, _P, _P, _P, _P,
                       C.c_size_t, _P]),
    "aicam_reid_crops": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _I, C.c_float, C.c_uint64,
                              C.c_uint64, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "aicam_reid_crops_nv12": (_I, [_P, _I, _I, _I, _P, _P, _P, _P, _I, C.c_float, C.c_uint64,
                                   C.c_uint64, _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    "aicam_tracker_create": (_I, [C.POINTER(TrackerConfig), C.POINTER(_P)]),
    "aicam_tracker_destroy": (None, [_P]),
    "aicam_tracker_reset": (_I, [_P, _P]),
    "aicam_tracker_reset_streams": (_I, [_P, _P, _P]),
    "aicam_tracker_set_stream_assoc": (_I, [_P, _P, C.POINTER(StreamAssoc), _I, _P]),
    "aicam_tracker_step": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "aicam_tracker_step_present": (_I, [_P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "aicam_tracker_cost_probe": (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "aicam_tracker_snapshot": (_I, [_P, _I, _P, _P, _I]),
    "aicam_tracker_overflow": (_I, [_P, _P]),
    "aicam_lsap": (_I, [_P, _I, _I, _I, _P, _P]),
    "aicam_kf_gating": (_I, [_P, _P, _I, _I, _P, _P]),
    "aicam_overlay_draw": (_I, [_P, _I, _I, _I, _P, _P, _P, _I, _I, _P]),
}

_lib = None


def load():
    """Load libaicam.so and bind every declared symbol.  Raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libaicam.so is not built (%s). Run `python -c 'import __graft_entry__ as g; "
                "g.build()'`; there is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code):
    if code != OK:
        raise AicamError(code, load().aicam_last_error().decode(errors="replace"))
    return code


def ptr(t):
    """Device/host address of a torch tensor or numpy array (None -> NULL)."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)


def stream_ptr(device=None):
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
