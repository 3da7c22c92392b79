"""ctypes binding of libb200track.so (include/b200track.h).

The library is the product: there is no Python / NumPy / CPU fallback behind it.  ``load()``
raises if the shared object has not been built (``python yolov7-tracker_b200/build.py``) and every
wrapper raises ``B2TError`` on a non-zero return code.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# B2T_LIB_PATH: diagnostic twin of the library (build.py --trace), never a different implementation
LIB_PATH = os.environ.get("B2T_LIB_PATH") or os.path.join(HERE, "libb200track.so")

F32, F64 = 0, 1
FMT_XYAH, FMT_XYWH, FMT_NSA = 0, 1, 2
SORT, BYTETRACK, BOTSORT, CBIOU = 0, 1, 2, 3
FLAG_MEAN_F32, FLAG_NOT_TRACKED = 1, 2
ACT_BF16, ACT_F16 = 0, 1
OUT_COLS, STAT_WORDS, STAT_PHASE0, STAT_SUB0 = 8, 64, 16, 32
GMC_STAT_WORDS, GMC_FIRST_FRAME, GMC_FEW_POINTS, GMC_TRUNCATED = 8, 1, 2, 4
(STAT_NOUT, STAT_NEXT_ID, STAT_NTRACKED, STAT_NLOST, STAT_ERR, STAT_FRAME, STAT_NPOOL, STAT_NBIRTH,
 STAT_NHI, STAT_NLO, STAT_NEDGE, STAT_NMATCH0) = range(12)
FMT_BY_NAME = {"default": FMT_XYAH, "botsort": FMT_XYWH, "strongsort": FMT_NSA}
KIND_BY_NAME = {"sort": SORT, "bytetrack": BYTETRACK, "botsort": BOTSORT, "c_biou": CBIOU}


class B2TError(RuntimeError):
    pass


class TrackerConfig(C.Structure):
    _fields_ = [("kind", C.c_int), ("dtype", C.c_int), ("fmt", C.c_int), ("n_seq", C.c_int), ("cap", C.c_int),
                ("dmax", C.c_int), ("ecap", C.c_int), ("use_gmc", C.c_int), ("track_buffer", C.c_int),
                ("conf_thresh", C.c_double), ("iou_thresh", C.c_double), ("frame_rate", C.c_double)]


class ConvDesc(C.Structure):
    _fields_ = [("x", C.c_void_p), ("w_packed", C.c_void_p), ("bias", C.c_void_p), ("y", C.c_void_p),
                ("n", C.c_int), ("h", C.c_int), ("w", C.c_int), ("cin", C.c_int), ("in_pitch", C.c_int), ("in_coff", C.c_int),
                ("cout", C.c_int), ("cout_rows", C.c_int), ("kh", C.c_int), ("kw", C.c_int), ("stride", C.c_int),
                ("out_pitch", C.c_int), ("out_coff", C.c_int), ("act", C.c_int), ("out_f32", C.c_int),
                ("block_n", C.c_int), ("tile_w", C.c_int), ("stages", C.c_int), ("in_row_pixels", C.c_int), ("rowpack", C.c_int), ("io_dtype", C.c_int),
                ("halo", C.c_int), ("halo_bufs", C.c_int), ("tps", C.c_int), ("kpair", C.c_int), ("out_bufs", C.c_int), ("mt", C.c_int), ("producers", C.c_int), ("splits", C.c_int)]


_P, _I, _D, _SZ = C.c_void_p, C.c_int, C.c_double, C.c_size_t

SIGNATURES = {
    "b2t_last_error": (C.c_char_p, []),
    "b2t_version": (_I, []),
    "b2t_launch_count": (C.c_longlong, []),
    "b2t_kalman_initiate": (_I, [_I, _I, _P, _P, _P, _I, _P]),
    "b2t_kalman_predict": (_I, [_I, _I, _P, _P, _P, _I, _I, _P]),
    "b2t_kalman_project": (_I, [_I, _I, _P, _P, _P, _P, _P, _P, _I, _P]),
    "b2t_kalman_update": (_I, [_I, _I, _P, _P, _P, _P, _P, _P, _I, _P]),
    "b2t_kalman_gating": (_I, [_I, _I, _P, _P, _P, _I, _I, _I, _P, _P]),
    "b2t_gmc_apply": (_I, [_I, _P, _P, _I, C.POINTER(C.c_double), _P]),
    "b2t_iou_cost": (_I, [_I, _P, _I, _P, _I, _P, _I, _I, _I, _P]),
    "b2t_lap_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "b2t_lap_solve": (_I, [_I, _P, _I, _I, _I, _D, _P, _P, _P, _SZ, _I, _P]),
    "b2t_tracker_state_bytes": (_SZ, [C.POINTER(TrackerConfig)]),
    "b2t_tracker_create": (_I, [C.POINTER(TrackerConfig), _P, _P, C.POINTER(_P)]),
    "b2t_tracker_reset": (_I, [_P, _P]),
    "b2t_tracker_destroy": (None, [_P]),
    "b2t_tracker_out_cols": (_I, []),
    "b2t_tracker_stat_words": (_I, []),
    "b2t_tracker_step": (_I, [_P, _P, _P, _P, _P, _P, _I, _P, _I, _P]),
    "b2t_tracker_step_host": (_I, [_P, _P, _P, _P, _P, _P, _I, _P, _I, _P]),
    "b2t_tracker_read_slot": (_I, [_P, _I, _I, _P, _P, _P]),
    "b2t_tracker_list_cols": (_I, []),
    "b2t_tracker_read_list": (_I, [_P, _I, _I, _P, _I, C.POINTER(C.c_int), _P]),
    "b2t_conv_last_error": (C.c_char_p, []),
    "b2t_conv_plan_create": (_I, [C.POINTER(ConvDesc), C.POINTER(_P)]),
    "b2t_conv_plan_destroy": (None, [_P]),
    "b2t_conv_plan_flops": (C.c_double, [_P]),
    "b2t_conv_plan_info": (_I, [_P, C.POINTER(C.c_int), _I]),
    "b2t_conv_run": (_I, [_P, _P]),
    "b2t_conv_plan_trace": (_I, [_P, C.POINTER(C.c_longlong), _I]),
    "b2t_detect_last_error": (C.c_char_p, []),
    "b2t_image_reorg": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "b2t_image_reorg_padded": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "b2t_upsample2x": (_I, [_P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P]),
    "b2t_spp_pool": (_I, [_P, _I, _I, _I, _I, _I, _I, _P]),
    "b2t_detect_decode": (_I, [_P, _I, _P, _I, _I, _I, _I, _I, C.c_longlong, C.c_longlong, C.c_float, C.POINTER(C.c_float), _P]),
    "b2t_nms_workspace_bytes": (_SZ, [_I, _I, _I]),
    "b2t_nms": (_I, [_P, _I, _I, _I, C.c_float, C.c_float, _I, _I, _I, _I, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                     _P, _SZ, _P, _P, _P]),
    "b2t_letterbox": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "b2t_letterbox_reorg": (_I, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _I, _I, _I, _P]),
    "b2t_gmc_workspace_bytes": (_SZ, [_I, _I, _I, _I, _I]),
    "b2t_gmc_reset": (_I, [_P, _I, _I, _I, _I, _I, _P]),
    "b2t_gmc_estimate": (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _I, C.c_float, _P, _I, _P, _P, _P]),
    "b2t_gmc_prepare": (_I, [_P, _I, _I, _I, _I, _I, _P, _I, _I, _P]),
    "b2t_gmc_estimate_prepared": (_I, [_I, _I, _I, _I, _P, _P, _I, C.c_float, _P, _I, _I, _P, _P, _P]),
    "b2t_gmc_workspace_layout": (_I, [_I, _I, _I, _I, _I, C.POINTER(_SZ), _I]),
    "b2t_reid_crops": (_I, [_P, _P, _I, _P, _I, _P]),
    "b2t_maxpool3x3s2": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "b2t_maxpool2x2s2": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "b2t_image_nhwc16": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "b2t_add_relu": (_I, [_P, _P, _P, C.c_longlong, _I, _P]),
    "b2t_batchnorm_batch_stats": (_I, [_P, _P, C.c_longlong, _I, _P, _P, C.c_float, _I, _P, _I, _P]),
    "b2t_avgpool_l2norm": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "b2t_detect_nms": (_I, [_P, _I, _I, _I, C.c_float, C.c_float, _I, _I, _I, _I, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                            _P, _SZ, _P, _P, _P]),
}


class HeadLevel(C.Structure):
    """include/b200track.h b2t_head_level"""
    _fields_ = [("raw", C.c_void_p), ("raw_pitch", C.c_int), ("h", C.c_int), ("w", C.c_int), ("stride", C.c_float),
                ("anchors", C.c_float * 6), ("level_off", C.c_longlong)]


# the NMS translation unit also compiles for the host simulator (tests/hostsim)
NMS_SYMBOLS = ["b2t_detect_last_error", "b2t_nms_workspace_bytes", "b2t_nms", "b2t_detect_nms", "b2t_letterbox", "b2t_letterbox_reorg",
               "b2t_gmc_workspace_bytes", "b2t_gmc_reset", "b2t_gmc_estimate", "b2t_gmc_workspace_layout", "b2t_gmc_prepare", "b2t_gmc_estimate_prepared"]

# the association branch (csrc/b2t_tracker.cu); the rest are the detector's translation units
TRACKER_SYMBOLS = [n for n in SIGNATURES if not n.startswith(("b2t_conv", "b2t_detect", "b2t_image", "b2t_upsample", "b2t_spp", "b2t_nms", "b2t_letterbox", "b2t_gmc_workspace", "b2t_gmc_reset", "b2t_gmc_estimate", "b2t_gmc_prepare",
                                                                   "b2t_reid", "b2t_maxpool", "b2t_add_relu", "b2t_avgpool", "b2t_batchnorm"))]


def act_dtype_code(torch_dtype):
    """torch.float16 / torch.bfloat16 -> B2T_ACT_F16 / B2T_ACT_BF16 (include/b200track.h)."""
    name = str(torch_dtype)
    if name == "torch.float16":
        return ACT_F16
    if name == "torch.bfloat16":
        return ACT_BF16
    raise B2TError("activation dtype must be torch.float16 or torch.bfloat16, got %s" % name)


def declare(lib, names=None):
    """Attach restype / argtypes for every symbol include/b200track.h declares (or the given subset)."""
    for name, (res, args) in SIGNATURES.items():
        if names is not None and name not in names:
            continue
        fn = getattr(lib, name)          # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2TError("libb200track.so is not built (%s). Run `python yolov7-tracker_b200/build.py`; "
                           "there is no CPU fallback." % LIB_PATH)
        _lib = declare(C.CDLL(LIB_PATH))
    return _lib


def check(lib, rc):
    if rc != 0:
        raise B2TError("libb200track error %d: %s" % (rc, (lib.b2t_last_error() or b"").decode()))
