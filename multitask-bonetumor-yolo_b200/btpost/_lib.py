"""ctypes binding of ``libbtpost.so`` (C ABI declared in ``include/btpost.h``).

There is no CPU or PyTorch fallback: if the shared library has not been built
(``make -C multitask-bonetumor-yolo_b200/csrc`` or ``__graft_entry__.build()``) loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_HERE = Path(__file__).resolve().parent
import os

# BTPOST_LIB lets developer scripts load the instrumented debug build (scripts/phase_timing.py)
LIB_PATH = Path(os.environ.get("BTPOST_LIB", _HERE / "libbtpost.so"))

BT_NUM_AREA = 4
BT_MAX_IOU_THRS = 16
BT_MAX_CURVE_THRS = 1024
LAYOUT_L2, LAYOUT_L1 = 0, 1
CLASS_AGNOSTIC, CLASS_AWARE, CLASS_OFFSET = 0, 1, 2
GT_LITERAL, GT_INTENDED = 0, 1
MASK_U8, MASK_F32 = 0, 1


class _IoMicro(C.Union):
    _fields_ = [("io_micro", C.c_int32), ("reserved", C.c_int32 * 1)]


class BtParams(C.Structure):
    _anonymous_ = ("_io_micro",)
    _fields_ = [
        ("batch", C.c_int32), ("num_anchors", C.c_int32), ("nc", C.c_int32), ("nm", C.c_int32),
        ("reg_max", C.c_int32), ("img_h", C.c_int32), ("img_w", C.c_int32),
        ("proto_h", C.c_int32), ("proto_w", C.c_int32), ("layout", C.c_int32),
        ("conf_thres", C.c_float), ("iou_thres", C.c_double),
        ("max_det", C.c_int32), ("max_cand", C.c_int32), ("class_mode", C.c_int32), ("max_wh", C.c_float),
        ("clamp_boxes", C.c_int32), ("gt_mode", C.c_int32), ("max_gt", C.c_int32), ("num_gt_rows", C.c_int32),
        ("iou_match_thresh", C.c_float), ("crop", C.c_int32), ("gt_mask_dtype", C.c_int32),
        ("proj_bias", C.c_float), ("num_iou_thrs", C.c_int32),
        ("iou_thrs", C.c_double * BT_MAX_IOU_THRS),
        ("image_offset", C.c_int32), ("nms_threads", C.c_int32), ("proto_dtype", C.c_int32), ("head_dtype", C.c_int32),
        ("drop_gt_no_cand", C.c_int32), ("in_flight", C.c_int32), ("io_soft_dice", C.c_int32), ("_io_micro", _IoMicro),
    ]


_IO_FIELDS = [
    "head", "maps0", "maps1", "maps2", "coeffs", "protos", "det_boxes_gt", "masks_gt", "proj_weight",
    "det_count", "dets", "det_keep", "det_anchor", "det_coeff", "n_cand",
    "gt_count", "gt_boxes", "gt_boxes_raw", "gt_labels",
    "cm", "seg_cnt4", "uni_cnt4",
    "cm_pos", "seg_img3", "seg_dice", "seg_iou", "uni_img3", "uni_dice", "uni_iou", "inst_area", "inst_inter",
    "seg_mask", "seg_logits", "uni_mask", "inst_bits", "inst_masks",
    "dt_match", "dt_ignore", "gt_ignore",
    "seg_prob_sum", "gt_rows_total", "sweep", "image_base", "seg_sweep",
]


class BtIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in _IO_FIELDS]


SOFT_DICE_FIELDS = ["seg_soft2", "seg_soft_dice", "seg_soft_acc"]


class BtIOSoftDice(BtIO):
    """A BtIO followed by the soft-Dice outputs (pass it with BtParams.io_soft_dice = 1)."""
    _fields_ = [(n, C.c_void_p) for n in SOFT_DICE_FIELDS]


class BtIOMicro(BtIOSoftDice):
    """A BtIOSoftDice followed by the class-agnostic sweep state (pass it with BtParams.io_micro = 1)."""
    _fields_ = [("micro_sweep", C.c_void_p)]


_lib = None


def load():
    """Load libbtpost.so; raises RuntimeError (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} not found: build the CUDA library first (make -C multitask-bonetumor-yolo_b200/csrc "
            "or python -c 'import __graft_entry__ as g; g.build()').  btpost has no CPU fallback.")
    L = C.CDLL(str(LIB_PATH))
    L.btpost_version.restype = C.c_int
    L.btpost_error_string.restype = C.c_char_p
    L.btpost_error_string.argtypes = [C.c_int]
    L.btpost_workspace_bytes.argtypes = [C.POINTER(BtParams), C.POINTER(C.c_size_t)]
    for name in ("btpost_decode_filter", "btpost_nms_match", "btpost_masks", "btpost_run"):
        f = getattr(L, name)
        f.argtypes = [C.POINTER(BtParams), C.POINTER(BtIO), C.c_void_p, C.c_size_t, C.c_void_p]
        f.restype = C.c_int
    L.btpost_synth_batch.argtypes = [C.c_int32] * 4 + [C.c_void_p] * 7
    L.btpost_synth_batch.restype = C.c_int
    L.btpost_masks_parts.argtypes = [C.POINTER(BtParams), C.POINTER(BtIO), C.c_void_p, C.c_size_t, C.c_void_p, C.c_int]
    L.btpost_masks_parts.restype = C.c_int
    L.btpost_sweep_bytes.argtypes = [C.c_int64, C.POINTER(C.c_size_t)]
    L.btpost_sweep_reset.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    L.btpost_sweep_accumulate_bytes.argtypes = [C.c_int64, C.POINTER(C.c_size_t)]
    L.btpost_sweep_accumulate.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                          C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_size_t, C.c_void_p]
    L.btpost_sweep_accumulate_ext.argtypes = (L.btpost_sweep_accumulate.argtypes[:13] + [C.c_void_p]
                                              + L.btpost_sweep_accumulate.argtypes[13:])   # + scores after recall
    L.btpost_surface_bytes.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]
    L.btpost_surface_distance.argtypes = [C.c_int32, C.c_int32] + [C.c_void_p] * 2 + [C.c_int32] + [C.c_void_p] * 5 + [C.c_size_t,
                                                                                                                      C.c_void_p]
    L.btpost_seg_curve.argtypes = [C.POINTER(BtParams), C.c_void_p, C.c_size_t, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]
    for name in ("btpost_sweep_bytes", "btpost_sweep_reset", "btpost_sweep_accumulate_bytes", "btpost_sweep_accumulate",
                 "btpost_sweep_accumulate_ext", "btpost_surface_bytes", "btpost_surface_distance", "btpost_seg_curve"):
        getattr(L, name).restype = C.c_int
    _lib = L
    return L


SWEEP_HEADER_I64 = 512
SWEEP_N_RECORDS, SWEEP_N_IMAGES, SWEEP_FSUM, SWEEP_CAPACITY, SWEEP_NPIG, SWEEP_USER = 0, 2, 3, 7, 8, 72
PROTO_F32, PROTO_BF16 = 0, 1
HEAD_F32, HEAD_BF16 = 0, 1
MASKS_PACK, MASKS_CONTRACT, MASKS_CELLS = 1, 2, 4   # btpost_masks_parts


def check(rc: int, what: str):
    if rc != 0:
        msg = load().btpost_error_string(rc).decode()
        exc = ValueError if rc in (-1, -2, -4) else RuntimeError
        raise exc(f"{what} failed: {msg} (code {rc})")
