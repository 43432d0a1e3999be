"""ctypes binding of libysb_postproc.so (C ABI in include/ysb_postproc.h).

The library is the product: if it is missing or cannot be loaded every op raises -- there is no
PyTorch/CPU fallback anywhere in this package.
"""
import ctypes
import os

PKG = os.path.dirname(os.path.abspath(__file__))
# YSB_LIBRARY: load another build of the same ABI (A/B runs of kernel experiments); default = the in-tree build
LIB_PATH = os.environ.get("YSB_LIBRARY") or os.path.join(PKG, "_lib", "libysb_postproc.so")

YSB_MAX_LEVELS = 8
YSB_MAX_ANCHORS = 9
YSB_MAX_DET_LIMIT = 1024
YSB_MAX_CANDIDATES = 4194303
YSB_MAX_CANDIDATES_WIDE = 2097151   # candidate limit when num_classes > 1024 (11-bit class field of the sort key)
YSB_MAX_CLASSES = 2048

# enum ysb_family
YOLOV5, YOLOV7, YOLOX, YOLOV8, RETINANET, RETINANET_EXP, FCOS = range(7)
FAMILY_IDS = {"yolov5": YOLOV5, "yolov7": YOLOV7, "yolox": YOLOX, "yolov8": YOLOV8, "retinanet": RETINANET,
              "retinanet_exp": RETINANET_EXP, "fcos": FCOS}
INPUT_RAW_HEADS, INPUT_DECODED_ROWS = 0, 1
INPUT_RAW_HEADS_NHWC = 2   # raw heads in channels-last memory (YOLOv5, YOLOX, YOLOv8, FCOS)
# enum ysb_dtype (element type of the raw heads)
DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2
DTYPE_F64 = 3   # ground truth of ysb_match_step only
IOU_NUMBA_F64MIX, IOU_F32, GIOU, DIOU, CIOU = range(5)
IOU_KIND_IDS = {"numba": IOU_NUMBA_F64MIX, "iou": IOU_F32, "giou": GIOU, "diou": DIOU, "ciou": CIOU}
CMP_GE, CMP_GT = 0, 1

ABI_VERSION = 6
YSB_MAX_PASSES = 4
YSB_MAX_PEERS = 16
YSB_IPC_HANDLE_BYTES = 64
YSB_CNT_ABSENT = -2   # gathered count of an image a rank did not have in a partial step
YSB_OK, YSB_ERR_BAD_ARG, YSB_ERR_UNSUPPORTED, YSB_ERR_WORKSPACE, YSB_ERR_CUDA, YSB_ERR_LIMIT = 0, -1, -2, -3, -4, -5


class YsbParams(ctypes.Structure):
    """Mirror of ``struct ysb_params``."""
    _fields_ = [
        ("family", ctypes.c_int32),
        ("input_kind", ctypes.c_int32),
        ("batch", ctypes.c_int32),
        ("num_classes", ctypes.c_int32),
        ("img_h", ctypes.c_int32),
        ("img_w", ctypes.c_int32),
        ("num_levels", ctypes.c_int32),
        ("level_h", ctypes.c_int32 * YSB_MAX_LEVELS),
        ("level_w", ctypes.c_int32 * YSB_MAX_LEVELS),
        ("level_stride", ctypes.c_float * YSB_MAX_LEVELS),
        ("anchors_per_cell", ctypes.c_int32),
        ("anchor", ((ctypes.c_float * 4) * YSB_MAX_ANCHORS) * YSB_MAX_LEVELS),
        ("reg_scale", ctypes.c_float * 4),
        ("dfl_bins", ctypes.c_int32),
        ("conf_thr", ctypes.c_float),
        ("cls_thr", ctypes.c_float),
        ("pre_nms_thr", ctypes.c_float),
        ("iou_thr", ctypes.c_double),
        ("max_det", ctypes.c_int32),
        ("class_aware", ctypes.c_int32),
        ("multi_label", ctypes.c_int32),
        ("postprocess_bbox", ctypes.c_int32),
        ("min_box_wh", ctypes.c_float),
        ("pre_nms_topk", ctypes.c_int32),
        ("thresh_with_ctr", ctypes.c_int32),
        ("decoded_rows", ctypes.c_int32),
        ("tta_scale", ctypes.c_float),
        ("tta_flip", ctypes.c_int32),
        ("tta_img_h", ctypes.c_int32),
        ("tta_img_w", ctypes.c_int32),
        ("d_letterbox", ctypes.c_void_p),
        ("head_dtype", ctypes.c_int32),
    ]


class YsbGather(ctypes.Structure):
    """Mirror of ``struct ysb_gather``."""
    _fields_ = [
        ("world", ctypes.c_int32),
        ("rank", ctypes.c_int32),
        ("slots", ctypes.c_int32),
        ("batch", ctypes.c_int32),
        ("max_det", ctypes.c_int32),
        ("d_buf", ctypes.c_void_p * YSB_MAX_PEERS),
    ]


class YsbMatchStep(ctypes.Structure):
    """Mirror of ``struct ysb_match_step``."""
    _fields_ = [
        ("world", ctypes.c_int32),
        ("batch", ctypes.c_int32),
        ("max_det", ctypes.c_int32),
        ("max_gt", ctypes.c_int32),
        ("d_rows", ctypes.c_void_p),
        ("rows_rank_bytes", ctypes.c_int64),
        ("d_cnt", ctypes.c_void_p),
        ("cnt_rank_bytes", ctypes.c_int64),
        ("d_gt", ctypes.c_void_p),
        ("d_gt_cnt", ctypes.c_void_p),
        ("gt_dtype", ctypes.c_int32),
    ]


class YsbError(RuntimeError):
    def __init__(self, status, what):
        self.status = status
        super().__init__(what)


_lib = None

_SIGNATURES = {
    "ysb_abi_version": (ctypes.c_int, []),
    "ysb_status_string": (ctypes.c_char_p, [ctypes.c_int]),
    "ysb_last_cuda_error": (ctypes.c_int, []),
    "ysb_num_candidates": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_int64),
                                          ctypes.POINTER(ctypes.c_int32)]),
    "ysb_decode": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                  ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_filter_candidates": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                             ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_select_nms": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                      ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_postprocess_workspace_bytes": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_postprocess": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_nms_workspace_bytes": (ctypes.c_int, [ctypes.c_int64, ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_nms": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_double, ctypes.c_int,
                               ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p,
                               ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_decode_into": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p]),
    "ysb_postprocess_tta_workspace_bytes": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.c_int,
                                                           ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_postprocess_tta": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                           ctypes.POINTER(ctypes.c_int32), ctypes.c_void_p, ctypes.c_size_t,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_filter_candidates_tta": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                                 ctypes.POINTER(ctypes.c_int32), ctypes.c_void_p, ctypes.c_int64,
                                                 ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_select_nms_tta": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                          ctypes.POINTER(ctypes.c_int32), ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                          ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_select_nms_tta_gather": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                                 ctypes.POINTER(ctypes.c_int32), ctypes.c_void_p, ctypes.c_int64,
                                                 ctypes.c_void_p, ctypes.POINTER(YsbGather), ctypes.c_int, ctypes.c_void_p,
                                                 ctypes.c_void_p]),
    "ysb_soft_nms": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_float, ctypes.c_int, ctypes.c_int,
                                    ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_undo_letterbox": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                          ctypes.c_void_p]),
    "ysb_pairwise_iou": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_elementwise_iou": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
                                           ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_elementwise_iou_backward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
                                                    ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                                    ctypes.c_void_p]),
    "ysb_pairwise_iou_backward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
                                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_wbf_workspace_bytes": (ctypes.c_int, [ctypes.c_int, ctypes.c_int64, ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_wbf": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double,
                               ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                               ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_wbf_collect": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                       ctypes.c_int, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_float), ctypes.c_int,
                                       ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "ysb_selftest_reciprocal": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_set_nms_cta_threads": (ctypes.c_int, [ctypes.c_int]),
    "ysb_map_iou": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                   ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_compute_tp_workspace_bytes": (ctypes.c_int, [ctypes.c_int64, ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_compute_tp": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_double),
                                      ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_match_tp_workspace_bytes": (ctypes.c_int, [ctypes.POINTER(YsbMatchStep), ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_match_tp": (ctypes.c_int, [ctypes.POINTER(YsbMatchStep), ctypes.POINTER(ctypes.c_double), ctypes.c_void_p,
                                    ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_match_compact": (ctypes.c_int, [ctypes.POINTER(YsbMatchStep), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                         ctypes.c_int64, ctypes.c_void_p]),
    "ysb_gather_buffer_bytes": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                               ctypes.POINTER(ctypes.c_size_t)]),
    "ysb_gather_alloc": (ctypes.c_int, [ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p]),
    "ysb_gather_open": (ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ysb_gather_close": (ctypes.c_int, [ctypes.c_void_p]),
    "ysb_gather_free": (ctypes.c_int, [ctypes.c_void_p]),
    "ysb_gather_slot_views": (ctypes.c_int, [ctypes.POINTER(YsbGather), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p),
                                             ctypes.POINTER(ctypes.c_void_p)]),
    "ysb_gather_strides": (ctypes.c_int, [ctypes.POINTER(YsbGather), ctypes.POINTER(ctypes.c_int64),
                                          ctypes.POINTER(ctypes.c_int64)]),
    "ysb_gather_begin": (ctypes.c_int, [ctypes.POINTER(YsbGather), ctypes.c_int, ctypes.c_void_p, ctypes.c_int64,
                                        ctypes.c_void_p]),
    "ysb_select_nms_gather": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p), ctypes.c_int,
                                             ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.POINTER(YsbGather),
                                             ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "ysb_select_nms_gather_partial": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.POINTER(ctypes.c_void_p),
                                                     ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                                     ctypes.POINTER(YsbGather), ctypes.c_int, ctypes.c_void_p,
                                                     ctypes.c_void_p]),
    "ysb_select_nms_tta_gather_partial": (ctypes.c_int, [ctypes.POINTER(YsbParams), ctypes.c_int,
                                                         ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int32),
                                                         ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p,
                                                         ctypes.POINTER(YsbGather), ctypes.c_int, ctypes.c_void_p,
                                                         ctypes.c_void_p]),
    "ysb_gather_wait": (ctypes.c_int, [ctypes.POINTER(YsbGather), ctypes.c_int, ctypes.c_void_p]),
    "ysb_gather_error": (ctypes.c_int, [ctypes.POINTER(YsbGather), ctypes.POINTER(ctypes.c_uint32)]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load():
    """Load the shared library (once).  Raises if it has not been built -- never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -m yoloseries_b200.build` "
                "(or __graft_entry__.build()); yoloseries_b200 has no CPU/PyTorch fallback")
        # RTLD_GLOBAL: the torch extension (libysb_torch.so, _ops.py) binds its ysb_* symbols to THIS library
        lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.ysb_abi_version() != ABI_VERSION:
            raise ImportError("libysb_postproc.so ABI version mismatch")
        _lib = lib
    return _lib


def check(status, what="ysb call"):
    """Map a ysb_status to the exception the reference's callers expect (SURVEY.md 8b conventions)."""
    if status == YSB_OK:
        return
    lib = load()
    msg = lib.ysb_status_string(status).decode()
    if status == YSB_ERR_CUDA:
        msg += f" [cudaError {lib.ysb_last_cuda_error()}]"
    if status in (YSB_ERR_BAD_ARG, YSB_ERR_LIMIT):
        raise ValueError(f"{what}: {msg}")
    if status == YSB_ERR_UNSUPPORTED:
        raise NotImplementedError(f"{what}: {msg}")
    raise YsbError(status, f"{what}: {msg}")


def unpack_keys(keys_u64, num_classes):
    """Sort keys written by ysb_filter_candidates -> (score float32, cand int64, cls int64).  The key layout depends on the
    call's class count (include/ysb_postproc.h): 10 class bits up to 1024 classes, 11 above."""
    import numpy as np
    cls_bits = 11 if num_classes > 1024 else 10
    cand_mask = (1 << (32 - cls_bits)) - 1
    cls_mask = (1 << cls_bits) - 1
    k = np.asarray(keys_u64).astype(np.uint64)
    score = (k >> np.uint64(32)).astype(np.uint32).view(np.float32)
    cand = cand_mask - ((k >> np.uint64(cls_bits)) & np.uint64(cand_mask)).astype(np.int64)
    cls = cls_mask - (k & np.uint64(cls_mask)).astype(np.int64)
    return score, cand, cls


def head_pointer_array(tensors):
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr
