"""Host-side mirror of the reference's post-processing / evaluation interface.

The reference has one operator boundary for this path (SURVEY.md §8b):

    map_preds, map_targets, det_log_preds, det_log_gts = \
        model._prepare_det_outputs_for_metrics_and_logging(det_outputs, det_boxes_gt, device, batch_size)

(`/root/reference/src/evaluate_model.py:174-178`; behaviour = `running_main_v2.py:720-882`), plus the
segmentation block `running_main_v2.py:672-713` and the output contract of `model(imgs, mode=...)`
(`main_modelv2.py:354-378`).  This module keeps those names, argument meanings, return formats and error
behaviour, and adds a batched `PostProcessor.run` that returns padded device tensors so the performance path
never builds ragged Python lists, and `Pipeline`, which keeps several batches in flight.  All arithmetic happens
in ``libbtpost.so`` (hand-written sm_100a CUDA) behind the C ABI of ``include/btpost.h``; PyTorch only owns the
device memory and the streams.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass, field

import torch

from . import _lib
from ._lib import BtIO, BtIOSoftDice, BtParams

# Module constants with the reference's names and defaults (running_main_v2.py:51-53); overridable.
CONF_TH = 0.05
NMS_IOU = 0.6
TOP_K = 300


def map_iou_thresholds():
    """fp32 linspace(0.5, 0.95, 10) widened to double (running_main_v2.py:247)."""
    return [float(v) for v in torch.linspace(0.5, 0.95, 10).tolist()]


def num_anchors(img_size: int) -> int:
    return sum((img_size // s) ** 2 for s in (8, 16, 32))


# ------------------------------------------------------------------------------------------------
# a1: unpacking what the model hands over
# ------------------------------------------------------------------------------------------------
def unpack_seg_outputs(seg_outputs, proto_ch: int = 32, strict: bool = True):
    """The reference's defensive unpack of the Segment head output (`running_main_v2.py:286-316`, `:672-681`,
    `evaluate_model.py:142-151`): a 3-tuple ``(det_maps, mask_coeffs, protos)`` (train mode, `main_modelv2.py:354-360`)
    or a 2-tuple ``(det_cat, (mask_coeffs, protos))`` (eval mode).  Returns ``(det, mask_coeffs, protos)``.

    ``strict=True`` raises the ValueErrors of `_multitask_loss` (`running_main_v2.py:299-316`); ``strict=False`` is the
    validation/eval variant that silently skips the seg block and returns ``protos = None`` (`:680-688`)."""
    det = coeffs = protos = None
    ok = False
    if isinstance(seg_outputs, (list, tuple)):
        if len(seg_outputs) == 3:
            det, coeffs, protos = seg_outputs
            ok = True
        elif len(seg_outputs) == 2 and isinstance(seg_outputs[1], (list, tuple)) and len(seg_outputs[1]) == 2:
            det, (coeffs, protos) = seg_outputs
            ok = True
    if not ok:
        if strict:
            n = len(seg_outputs) if isinstance(seg_outputs, (list, tuple)) else type(seg_outputs)
            raise ValueError("Critical Error: seg_head_outputs has an unhandled structure. Expected 3-element tuple "
                             "(det_internal, mask_coeffs_3D_or_protos_3D, protos_4D) OR 2-element tuple "
                             f"(det_internal, (mask_coeffs_3D, protos_4D)). Got length {n}.")
        return None, None, None
    if not (isinstance(protos, torch.Tensor) and protos.ndim == 4):
        if strict:
            got = protos.shape if isinstance(protos, torch.Tensor) else type(protos)
            raise ValueError(f"actual_protos_tensor for seg_proto_projector must be 4D. Got shape: {got}. "
                             "This was derived from seg_head_outputs.")
        return det, coeffs, None
    if protos.shape[1] != proto_ch:
        if strict:
            raise ValueError(f"actual_protos_tensor channel mismatch. Expected {proto_ch}, got {protos.shape[1]}. "
                             f"Shape: {protos.shape}")
        return det, coeffs, None
    return det, coeffs, protos


def unpack_infer_dict(out_dict, nc: int = 3, proto_ch: int = 32):
    """What `ConvNeXtBiFPNYOLO.forward(x, mode="infer")` returns (`main_modelv2.py:362-378`): ``segment_preds_cat``
    ``[B, 4+nc+nm, N]`` and ``segment_protos`` = whatever the Ultralytics eval forward returned second (the 4-D prototype
    tensor, ``(mask_coeffs, protos)`` or ``(feats, mask_coeffs, protos)``).  Returns ``(head, protos)``."""
    if not isinstance(out_dict, dict) or "segment_preds_cat" not in out_dict or "segment_protos" not in out_dict:
        raise ValueError("postprocess_infer expects the dict of model(imgs, mode='infer') with the keys "
                         "'segment_preds_cat' and 'segment_protos' (main_modelv2.py:369-377)")
    head, protos = out_dict["segment_preds_cat"], out_dict["segment_protos"]
    if isinstance(protos, (list, tuple)):
        protos = protos[-1]
    if not (isinstance(protos, torch.Tensor) and protos.ndim == 4):
        got = protos.shape if isinstance(protos, torch.Tensor) else type(protos)
        raise ValueError(f"actual_protos_tensor for seg_proto_projector must be 4D. Got shape: {got}.")
    if protos.shape[1] != proto_ch:
        raise ValueError(f"actual_protos_tensor channel mismatch. Expected {proto_ch}, got {protos.shape[1]}. Shape: {protos.shape}")
    if not (isinstance(head, torch.Tensor) and head.ndim == 3 and head.shape[1] == 4 + nc + proto_ch):
        got = tuple(head.shape) if isinstance(head, torch.Tensor) else type(head)
        raise ValueError(f"segment_preds_cat must be [B, 4+nc+nm = {4 + nc + proto_ch}, N]. Got {got}.")
    return head, protos


@dataclass
class PostConfig:
    batch: int
    img_size: int = 640
    nc: int = 3
    nm: int = 32
    reg_max: int = 16
    conf_thres: float | None = None      # None -> module CONF_TH at call time
    iou_thres: float | None = None       # None -> module NMS_IOU
    max_det: int | None = None           # None -> module TOP_K
    max_cand: int = 0                    # Ultralytics max_nms: best-scoring candidates that enter the NMS (0 = all)
    class_mode: int = _lib.CLASS_AGNOSTIC
    max_wh: float = 7680.0
    clamp_boxes: bool = True
    gt_mode: int = _lib.GT_LITERAL
    max_gt: int = 32
    iou_match_thresh: float = 0.5
    crop: bool = True
    layout: int = _lib.LAYOUT_L2
    gt_mask_dtype: int = _lib.MASK_U8
    iou_thrs: list = field(default_factory=map_iou_thresholds)
    drop_gt_no_cand: bool = False        # True = v2 (running_main_v2.py:797-814): no candidate above CONF_TH -> empty target;
                                         # False = v3 (running_main_v3.py:541-571, canonical): the target is kept
    # optional dense outputs
    with_seg_mask: bool = False
    with_seg_logits: bool = False
    with_uni_mask: bool = False
    with_inst_masks: str | None = None   # None, "bits" ([B,K,S,S/8] bit-packed) or "dense" (+ [B,K,S,S] bytes)
    with_coco: bool = True
    with_seg_map: bool = False           # v3 segmentation-mAP prep (score numerator per image)
    with_soft_dice: bool = False         # v3 soft Dice on the projector probabilities: seg_soft2 / seg_soft_dice (+ seg_soft_acc)
    num_anchors: int | None = None
    nms_threads: int = 0                 # 0 = auto; 512 / 1024 force a variant of the NMS kernel
    in_flight: int = 0                   # batches kept in flight on the device (Pipeline sets its depth): grid sizes of the mask stage
    proto_bf16: bool = False             # prototypes arrive as torch.bfloat16 (widened exactly in the kernel)
    head_bf16: bool = False              # same for the L2 head tensor / the L1 raw maps


class PostProcessor:
    """Owns params, workspace and output tensors for one (batch, shape) configuration on one GPU."""

    def __init__(self, cfg: PostConfig, device="cuda:0", shared_counters: dict | None = None, sweep=None):
        self.lib = _lib.load()
        self.cfg = cfg
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("btpost runs on CUDA devices only (sm_100a); there is no CPU path")
        if cfg.with_inst_masks not in (None, "bits", "dense"):
            raise ValueError("with_inst_masks must be None, 'bits' or 'dense'")
        B, S = cfg.batch, cfg.img_size
        K = cfg.max_det if cfg.max_det is not None else TOP_K
        N = cfg.num_anchors if cfg.num_anchors is not None else num_anchors(S)
        self.B, self.S, self.K, self.N = B, S, K, N
        p = BtParams()
        p.batch, p.num_anchors, p.nc, p.nm, p.reg_max = B, N, cfg.nc, cfg.nm, cfg.reg_max
        p.img_h = p.img_w = S
        p.proto_h = p.proto_w = S // 4
        p.layout = cfg.layout
        p.conf_thres = cfg.conf_thres if cfg.conf_thres is not None else CONF_TH
        p.iou_thres = cfg.iou_thres if cfg.iou_thres is not None else NMS_IOU
        p.max_det, p.max_cand, p.class_mode, p.max_wh = K, cfg.max_cand, cfg.class_mode, cfg.max_wh
        p.clamp_boxes, p.gt_mode, p.max_gt = int(cfg.clamp_boxes), cfg.gt_mode, cfg.max_gt
        p.iou_match_thresh, p.crop, p.gt_mask_dtype = cfg.iou_match_thresh, int(cfg.crop), cfg.gt_mask_dtype
        p.num_iou_thrs = len(cfg.iou_thrs)
        p.nms_threads = cfg.nms_threads
        p.in_flight = cfg.in_flight
        p.proto_dtype = _lib.PROTO_BF16 if cfg.proto_bf16 else _lib.PROTO_F32
        p.head_dtype = _lib.HEAD_BF16 if cfg.head_bf16 else _lib.HEAD_F32
        p.drop_gt_no_cand = int(cfg.drop_gt_no_cand)
        p.io_soft_dice = int(cfg.with_soft_dice)   # the outputs below then travel in a BtIOSoftDice
        for i, v in enumerate(cfg.iou_thrs):
            p.iou_thrs[i] = v
        self.params = p
        nbytes = C.c_size_t()
        _lib.check(self.lib.btpost_workspace_bytes(C.byref(p), C.byref(nbytes)), "btpost_workspace_bytes")
        dev = self.device
        self.workspace = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=dev)
        self._ws_ptr = (self.workspace.data_ptr() + 255) // 256 * 256
        self._ws_bytes = nbytes.value
        G, A, T, nc, nm = cfg.max_gt, _lib.BT_NUM_AREA, len(cfg.iou_thrs), cfg.nc, cfg.nm
        z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)
        o = {
            "det_count": z(B, dtype=torch.int32), "dets": z(B, K, 6, dtype=torch.float32),
            "det_keep": z(B, K, dtype=torch.int64), "det_anchor": z(B, K, dtype=torch.int32),
            "det_coeff": z(B, K, nm, dtype=torch.float32), "n_cand": z(B, dtype=torch.int32),
            "gt_count": z(B, dtype=torch.int32), "gt_boxes": z(B, G, 4, dtype=torch.float32),
            "gt_boxes_raw": z(B, G, 4, dtype=torch.float32), "gt_labels": z(B, G, dtype=torch.int32),
            "gt_rows_total": z(B, dtype=torch.int32),
            "cm": z(nc, nc, dtype=torch.int64), "seg_cnt4": z(4, dtype=torch.int64), "uni_cnt4": z(4, dtype=torch.int64),
            "cm_pos": z(B, dtype=torch.int32), "seg_img3": z(B, 3, dtype=torch.int64),
            "seg_dice": z(B, dtype=torch.float32), "seg_iou": z(B, dtype=torch.float32),
            "uni_img3": z(B, 3, dtype=torch.int64), "uni_dice": z(B, dtype=torch.float32),
            "uni_iou": z(B, dtype=torch.float32), "inst_area": z(B, K, dtype=torch.int32),
            "inst_inter": z(B, K, dtype=torch.int32),
        }
        if sweep is not None and not shared_counters:
            shared_counters = sweep.counters()   # the accumulators live in the sweep header: one all-reduce merges everything
        if cfg.with_soft_dice:
            o["seg_soft2"] = z(B, 2, dtype=torch.int64)
            o["seg_soft_dice"] = z(B, dtype=torch.float32)
            o["seg_soft_acc"] = z(2, dtype=torch.int64)
        if shared_counters:   # Pipeline: every slot adds into the same accumulators (device atomics)
            for k in ("cm", "seg_cnt4", "uni_cnt4") + (("seg_soft_acc",) if cfg.with_soft_dice else ()):
                o[k] = shared_counters[k]
        if cfg.with_seg_mask:
            o["seg_mask"] = z(B, S, S, dtype=torch.uint8)
        if cfg.with_seg_logits:
            o["seg_logits"] = z(B, S, S, dtype=torch.float32)
        if cfg.with_uni_mask:
            o["uni_mask"] = z(B, S, S, dtype=torch.uint8)
        if cfg.with_inst_masks:
            o["inst_bits"] = z(B, K, S, S // 8, dtype=torch.uint8)
            if cfg.with_inst_masks == "dense":
                o["inst_masks"] = z(B, K, S, S, dtype=torch.uint8)
        if cfg.with_coco:
            o["dt_match"] = z(B, A, T, K, dtype=torch.int32)
            o["dt_ignore"] = z(B, A, T, K, dtype=torch.uint8)
            o["gt_ignore"] = z(B, A, G, dtype=torch.uint8)
        if cfg.with_seg_map:
            o["seg_prob_sum"] = z(B, dtype=torch.float64)
        self.out = o
        self.sweep = sweep                # a btpost.sweep.DeviceSweep: records are appended by the library itself
        if sweep is not None and not cfg.with_coco:
            raise ValueError("a sweep needs with_coco=True (the records are written by the COCO matching)")
        if sweep is not None and sweep.seg_ptr is not None and not cfg.with_seg_map:
            raise ValueError("a sweep with a segmentation-mAP ring (seg_map_capacity > 0) needs with_seg_map=True "
                             "(the records are scored with the mask kernel's seg_prob_sum)")
        if sweep is not None and sweep.soft_dice and not cfg.with_soft_dice:
            raise ValueError("a sweep with soft_dice=True needs with_soft_dice=True (the mask kernel adds the per-image "
                             "soft Dice into the sweep's seg_soft_acc)")
        self._empty_gt = torch.zeros(1, 6, dtype=torch.float32, device=dev)
        self.image_base = torch.zeros(1, dtype=torch.int32, device=dev)   # global index of image 0, read by the kernels

    # -- metric state ---------------------------------------------------------------------------
    def reset_metrics(self):
        """Zero the accumulated counters (confusion matrix, global pixel tp/fp/fn/tn, soft-Dice sum and count)."""
        for k in ("cm", "seg_cnt4", "uni_cnt4", "seg_soft_acc"):
            if k in self.out:
                self.out[k].zero_()

    def check_gt_overflow(self):
        """Raises when an image of the last batch had more GT rows than ``max_gt`` (the reference has no limit; the
        kernels drop the excess rows).  One device->host read of [B] counters."""
        tot = self.out["gt_rows_total"].cpu()
        if int(tot.max()) > self.cfg.max_gt:
            b = int(tot.argmax())
            raise ValueError(f"image {b} has {int(tot[b])} ground-truth rows, more than max_gt={self.cfg.max_gt}: "
                             "raise PostConfig.max_gt (<= 32)")

    # -- launch ---------------------------------------------------------------------------------
    def _check_in(self, t, shape, dtype, name):
        if t.device != self.device or t.dtype != dtype or tuple(t.shape) != tuple(shape) or not t.is_contiguous():
            raise ValueError(f"{name}: expected contiguous {dtype} {tuple(shape)} on {self.device}, "
                             f"got {t.dtype} {tuple(t.shape)} on {t.device}")

    def _io(self, head, protos, det_boxes_gt, masks_gt, proj_weight, maps=None, coeffs=None):
        io = BtIOSoftDice() if self.cfg.with_soft_dice else BtIO()
        cfg, B, S, N = self.cfg, self.B, self.S, self.N
        hdt = torch.bfloat16 if cfg.head_bf16 else torch.float32
        if cfg.layout == _lib.LAYOUT_L2:
            self._check_in(head, (B, 4 + cfg.nc + cfg.nm, N), hdt, "head")
            io.head = head.data_ptr()
        else:
            if maps is None or len(maps) != 3:
                raise ValueError("L1 layout: `maps` must be the list of 3 raw maps [B, 4*reg_max+nc, H_l, W_l]")
            for l, (m, s) in enumerate(zip(maps, (8, 16, 32))):
                self._check_in(m, (B, 4 * cfg.reg_max + cfg.nc, S // s, S // s), hdt, f"maps[{l}]")
                setattr(io, f"maps{l}", m.data_ptr())
            if coeffs is not None:
                self._check_in(coeffs, (B, cfg.nm, N), hdt, "coeffs")
                io.coeffs = coeffs.data_ptr()
        self._check_in(protos, (B, cfg.nm, S // 4, S // 4), torch.bfloat16 if cfg.proto_bf16 else torch.float32, "protos")
        io.protos = protos.data_ptr()
        if det_boxes_gt is None or det_boxes_gt.numel() == 0:
            det_boxes_gt, rows = self._empty_gt, 0
        else:
            rows = det_boxes_gt.shape[0]
            self._check_in(det_boxes_gt, (rows, 6), torch.float32, "det_boxes_gt")
        io.det_boxes_gt = det_boxes_gt.data_ptr()
        self.params.num_gt_rows = rows
        mdt = torch.uint8 if cfg.gt_mask_dtype == _lib.MASK_U8 else torch.float32
        if masks_gt.dim() == 3:
            masks_gt = masks_gt.unsqueeze(1)
        self._check_in(masks_gt, (B, 1, S, S), mdt, "masks_gt")
        io.masks_gt = masks_gt.data_ptr()
        self._check_in(proj_weight, (cfg.nm,), torch.float32, "proj_weight")
        io.proj_weight = proj_weight.data_ptr()
        for k, v in self.out.items():
            setattr(io, k, v.data_ptr())
        if self.sweep is not None:
            io.sweep = self.sweep.ptr
            io.seg_sweep = self.sweep.seg_ptr
            io.image_base = self.image_base.data_ptr()
        self._keepalive = (head, protos, det_boxes_gt, masks_gt, proj_weight, maps, coeffs)
        return io

    def run(self, head, protos, det_boxes_gt, masks_gt, proj_weight, proj_bias=0.0, *, maps=None, coeffs=None,
            stage="run", stream=None, image_offset=0):
        """Enqueue the hot path for one batch on the current (or given) CUDA stream; returns the
        dict of output tensors (device, padded to ``max_det`` / ``max_gt``; see include/btpost.h)."""
        # module constants are read at call time, as the reference reads its globals inside the loop
        if self.cfg.conf_thres is None:
            self.params.conf_thres = CONF_TH
        if self.cfg.iou_thres is None:
            self.params.iou_thres = NMS_IOU
        self.params.proj_bias = float(proj_bias)
        self.params.image_offset = int(image_offset)   # plus self.image_base[0] (device; what captured steps vary)
        io = self._io(head, protos, det_boxes_gt, masks_gt, proj_weight, maps, coeffs)
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        parts = {"masks_pack": _lib.MASKS_PACK, "masks_contract": _lib.MASKS_CONTRACT, "masks_cells": _lib.MASKS_CELLS}.get(stage)
        with torch.cuda.device(self.device):
            if parts is not None:   # one kernel group of the mask stage (bench.py times the HBM-side kernel alone)
                rc = self.lib.btpost_masks_parts(C.byref(self.params), C.byref(io), C.c_void_p(self._ws_ptr),
                                                 C.c_size_t(self._ws_bytes), C.c_void_p(st.cuda_stream), C.c_int(parts))
            else:
                fn = getattr(self.lib, f"btpost_{stage}")
                rc = fn(C.byref(self.params), C.byref(io), C.c_void_p(self._ws_ptr), C.c_size_t(self._ws_bytes),
                        C.c_void_p(st.cuda_stream))
        _lib.check(rc, f"btpost_{stage}")
        return self.out

    def capture(self, head, protos, det_boxes_gt, masks_gt, proj_weight, proj_bias=0.0, image_stride=0, **kw):
        """Capture one step on these (static) buffers into a CUDA graph; returns the graph, whose
        ``replay()`` re-runs the whole hot path with one host call (the library is capture-safe:
        no allocation, no synchronisation, caller's stream only).  ``image_stride`` > 0: every replay first adds it to
        the device-resident ``image_base`` (global index of the batch's first image in the sweep records), so a
        round-robin of slots numbers its images without any host work per step."""
        self.run(head, protos, det_boxes_gt, masks_gt, proj_weight, proj_bias, **kw)   # warm-up: attributes, module load
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            if image_stride:
                self.image_base.add_(int(image_stride))
            self.run(head, protos, det_boxes_gt, masks_gt, proj_weight, proj_bias, **kw)
        return g

    # -- reference-shaped views -----------------------------------------------------------------
    def to_reference_lists(self, out=None):
        """(map_preds, map_targets, det_log_preds, det_log_gts) exactly as
        `running_main_v2.py:720-882` builds them: CPU dicts for torchmetrics, device [K,6]/[G,5]
        tensors for `log_det_examples` (`multitask_logging.py:216,240`)."""
        o = out or self.out
        counts = o["det_count"].cpu().tolist()       # one D->H sync for the whole batch
        gcounts = o["gt_count"].cpu().tolist()
        ncand = o["n_cand"].cpu().tolist()
        if "gt_rows_total" in o:
            self.check_gt_overflow()
        dets_cpu, gtb_cpu, gtl_cpu = o["dets"].cpu(), o["gt_boxes"].cpu(), o["gt_labels"].cpu()
        map_preds, map_targets, log_preds, log_gts = [], [], [], []
        for b in range(self.B):
            k, g = counts[b], gcounts[b]
            if ncand[b] == 0 and self.cfg.drop_gt_no_cand:
                # v2 appends an empty target too when no box passes CONF_TH (running_main_v2.py:797-814)
                g = 0
            d = dets_cpu[b, :k]
            map_preds.append({"boxes": d[:, :4].clone(), "scores": d[:, 4].clone(), "labels": d[:, 5].long()})
            log_preds.append(o["dets"][b, :k])
            map_targets.append({"boxes": gtb_cpu[b, :g].clone(), "labels": gtl_cpu[b, :g].long()})
            log_gts.append(torch.cat([o["gt_boxes"][b, :g], o["gt_labels"][b, :g].float().unsqueeze(1)], dim=1))
        return map_preds, map_targets, log_preds, log_gts


class Pipeline:
    """``depth`` slots, each a PostProcessor with its OWN static input buffers, workspace and outputs, whose captured
    step is replayed on the slot's own stream: consecutive batches overlap on the GPU, so the NMS of batch i+1 (one CTA
    per image, most SMs idle) runs under the mask kernels of batch i.

    ``submit(head, protos, det_boxes_gt, masks_gt)`` copies one batch (device or pinned host tensors) into the next
    slot's input buffers on that slot's stream and replays its step; a producer can instead write straight into
    ``inputs[slot]`` and call ``replay(slot)`` (zero-copy).  ``wait(slot)`` blocks the host until the slot's step is
    done and returns its outputs, which stay valid until the slot is used again (``depth`` steps later).  The
    accumulated counters (cm, seg_cnt4, uni_cnt4, seg_soft_acc) are shared by all slots (device atomics):
    ``counters(key)``.

    ``det_boxes_gt`` lives in a fixed ``[gt_rows_cap, 6]`` buffer per slot; unused rows carry batch index -1, which
    matches no image."""

    def __init__(self, cfg: PostConfig, device="cuda:0", depth: int = 2, gt_rows_cap: int | None = None,
                 proj_weight=None, proj_bias: float = 0.0, sweep=None, auto_image_offset: bool = False):
        conf = cfg.conf_thres if cfg.conf_thres is not None else CONF_TH
        if depth > 1 and cfg.nms_threads == 0 and conf >= 0.01:
            # small-footprint NMS kernel: its CTAs share SMs with the mask kernels of the other batches in flight
            # (dense candidate lists keep the 1024-thread variant, which sorts them in registers)
            cfg = dataclasses.replace(cfg, nms_threads=512)
        if depth > 1 and cfg.in_flight == 0:
            cfg = dataclasses.replace(cfg, in_flight=depth)   # the mask stage's persistent kernels leave room for the other batches
        if cfg.layout != _lib.LAYOUT_L2:
            raise ValueError("Pipeline takes the L2 head layout ([B, 4+nc+nm, N])")
        self.cfg, self.depth = cfg, depth
        self.auto_image_offset = bool(auto_image_offset)   # images numbered on the device (see set_image_base)
        self.device = dev = torch.device(device)
        nc, B, S = cfg.nc, cfg.batch, cfg.img_size
        self.sweep = sweep
        self.shared = sweep.counters() if sweep is not None else {
            "cm": torch.zeros(nc, nc, dtype=torch.int64, device=dev), "seg_cnt4": torch.zeros(4, dtype=torch.int64, device=dev),
            "uni_cnt4": torch.zeros(4, dtype=torch.int64, device=dev), "seg_soft_acc": torch.zeros(2, dtype=torch.int64, device=dev)}
        self.procs = [PostProcessor(cfg, dev, shared_counters=self.shared, sweep=sweep) for _ in range(depth)]
        N = self.procs[0].N
        self.gt_rows_cap = gt_rows_cap if gt_rows_cap is not None else 4 * B
        hdt = torch.bfloat16 if cfg.head_bf16 else torch.float32
        pdt = torch.bfloat16 if cfg.proto_bf16 else torch.float32
        mdt = torch.uint8 if cfg.gt_mask_dtype == _lib.MASK_U8 else torch.float32
        self.inputs = []
        for _ in range(depth):
            gt = torch.zeros(self.gt_rows_cap, 6, dtype=torch.float32, device=dev)
            gt[:, 0] = -1.0
            self.inputs.append({"head": torch.zeros(B, 4 + nc + cfg.nm, N, dtype=hdt, device=dev),
                                "protos": torch.zeros(B, cfg.nm, S // 4, S // 4, dtype=pdt, device=dev),
                                "det_boxes_gt": gt,
                                "masks_gt": torch.zeros(B, 1, S, S, dtype=mdt, device=dev)})
        self.proj_weight = (proj_weight if proj_weight is not None else torch.zeros(cfg.nm)).to(dev, torch.float32).contiguous()
        self.proj_bias = float(proj_bias)
        self.streams = [torch.cuda.Stream(dev) for _ in range(depth)]
        self.events = [torch.cuda.Event() for _ in range(depth)]
        self.graphs = []
        self._i = 0
        self._capture()

    def _capture(self):
        self.graphs = []
        for p, inp in zip(self.procs, self.inputs):
            self.graphs.append(p.capture(inp["head"], inp["protos"], inp["det_boxes_gt"], inp["masks_gt"], self.proj_weight,
                                         self.proj_bias, image_stride=self.depth * self.cfg.batch if self.auto_image_offset else 0))
        self.reset_metrics()   # the warm-up / capture runs counted the zero inputs
        if self.auto_image_offset:
            self.set_image_base(0)
        torch.cuda.synchronize(self.device)
        self._bind_graphs()

    def _bind_graphs(self):
        """Raw executable-graph handles: a replay is then ONE cudaGraphLaunch on the slot's stream (a few microseconds of
        host time instead of a stream context manager around CUDAGraph.replay(); with five batches in flight the host has
        to get five launches out before the GPU is full).  Falls back to CUDAGraph.replay() when this torch build does
        not expose the handles."""
        self._exec, self._cudart = None, None
        try:
            rt = C.CDLL("libcudart.so.12")
            rt.cudaGraphLaunch.argtypes = [C.c_void_p, C.c_void_p]
            rt.cudaGraphLaunch.restype = C.c_int
            self._exec = [int(g.raw_cuda_graph_exec()) for g in self.graphs]
            self._cudart = rt
        except Exception:
            self._exec, self._cudart = None, None

    def set_image_base(self, first: int):
        """auto_image_offset: the next replayed step holds the images first .. first + B - 1, the one after it the
        next B, and so on (each slot's captured step adds depth * B to its own counter before it runs)."""
        if not self.auto_image_offset:
            raise ValueError("Pipeline was built without auto_image_offset")
        B, d = self.cfg.batch, self.depth
        for s, p in enumerate(self.procs):
            p.image_base.fill_(int(first) + ((s - self._i) % d) * B - d * B)

    # -- feeding --------------------------------------------------------------------------------
    def load(self, slot, head, protos, det_boxes_gt, masks_gt, stream=None):
        """Copy one batch into the slot's static input buffers (on `stream`, default: the slot's stream)."""
        inp = self.inputs[slot]
        st = stream if stream is not None else self.streams[slot]
        rows = 0 if det_boxes_gt is None else int(det_boxes_gt.shape[0])
        if rows > self.gt_rows_cap:
            raise ValueError(f"det_boxes_gt has {rows} rows, more than gt_rows_cap={self.gt_rows_cap}")
        with torch.cuda.stream(st):
            inp["head"].copy_(head, non_blocking=True)
            inp["protos"].copy_(protos, non_blocking=True)
            inp["masks_gt"].copy_(masks_gt.reshape(inp["masks_gt"].shape), non_blocking=True)
            if rows:
                inp["det_boxes_gt"][:rows].copy_(det_boxes_gt, non_blocking=True)
            inp["det_boxes_gt"][rows:, 0] = -1.0

    def fork(self):
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            st.wait_stream(cur)

    def replay(self, slot=None, image_offset=None):
        """Run the captured step of `slot` (default: round robin) on its stream; returns the slot's PostProcessor.
        `image_offset` = global index of the batch's first image (sweep records; one 4-byte fill on the slot's stream);
        a pipeline built with ``auto_image_offset`` numbers the images itself (round-robin replays only)."""
        i = self._i % self.depth if slot is None else slot
        self._i += 1
        if self.auto_image_offset and (image_offset is not None or slot is not None):
            raise ValueError("auto_image_offset: replay() takes neither a slot nor an image offset")
        st = self.streams[i]
        if image_offset is not None:
            with torch.cuda.stream(st):
                self.procs[i].image_base.fill_(int(image_offset))
        if self._exec is not None:
            rc = self._cudart.cudaGraphLaunch(self._exec[i], st.cuda_stream)
            if rc != 0:
                raise RuntimeError(f"cudaGraphLaunch failed with CUDA error {rc}")
        else:
            with torch.cuda.stream(st):
                self.graphs[i].replay()
        self.events[i].record(st)
        return self.procs[i]

    def submit(self, head, protos, det_boxes_gt, masks_gt, image_offset=None):
        """Copy one batch into the next slot and run it; returns the slot index (pass it to `wait`)."""
        i = self._i % self.depth
        self.load(i, head, protos, det_boxes_gt, masks_gt)
        self.replay(None if self.auto_image_offset else i, image_offset)
        return i

    def wait(self, slot):
        self.events[slot].synchronize()
        return self.procs[slot].out

    def join(self):
        cur = torch.cuda.current_stream(self.device)
        for st in self.streams:
            cur.wait_stream(st)

    def reset_metrics(self):
        if self.sweep is not None:
            self.sweep.reset()     # the shared counters live inside the sweep header
        else:
            for k in self.shared:
                self.shared[k].zero_()

    def counters(self, key):
        return self.shared[key]


_cached: dict = {}


def prepare_det_outputs_for_metrics_and_logging(det_outputs, det_boxes_gt, device, batch_size, *, img_size=640,
                                                nc=3, variant="v2"):
    """Drop-in for ``MultiTaskLitModel._prepare_det_outputs_for_metrics_and_logging``
    (`/root/reference/src/evaluate_model.py:174-178`).

    ``det_outputs`` is either the reference's list of three raw maps ``[B, 4*16+nc, H_l, W_l]`` (L1; fp32 or the
    bf16 a ``bf16-mixed`` forward produces) or the concatenated ``[B, 4+nc+32, N]`` tensor (L2, ``segment_preds_cat``).
    Returns ``(map_preds, map_targets, det_log_preds, det_log_gts)`` in the reference's formats.  ``variant="v2"``
    follows `running_main_v2.py:797-814` (an image without any candidate above CONF_TH gets an empty target),
    ``"v3"`` follows `running_main_v3.py:541-571` (target kept).  Only the detection stages run (decode/filter +
    NMS/matching); the mask stage needs prototypes and is reached through ``PostProcessor.run`` / ``postprocess_infer``.
    """
    if variant not in ("v2", "v3"):
        raise ValueError("variant must be 'v2' or 'v3'")
    device = torch.device(device)
    l1 = isinstance(det_outputs, (list, tuple))
    first = det_outputs[0] if l1 else det_outputs
    bf16 = first.dtype == torch.bfloat16
    key = (batch_size, img_size, nc, l1, bf16, str(device), CONF_TH, NMS_IOU, TOP_K, variant)
    pp = _cached.get(key)
    if pp is None:
        cfg = PostConfig(batch=batch_size, img_size=img_size, nc=nc, head_bf16=bf16, drop_gt_no_cand=(variant == "v2"),
                         layout=_lib.LAYOUT_L1 if l1 else _lib.LAYOUT_L2)
        pp = _cached[key] = PostProcessor(cfg, device)
        S = img_size
        pp._dummy_protos = torch.zeros(batch_size, 32, S // 4, S // 4, device=device)
        pp._dummy_masks = torch.zeros(batch_size, 1, S, S, dtype=torch.uint8, device=device)
        pp._dummy_w = torch.zeros(32, device=device)
        pp._dummy_coeffs = torch.zeros(batch_size, 32, pp.N, device=device, dtype=torch.bfloat16 if bf16 else torch.float32)
    dt = torch.bfloat16 if bf16 else torch.float32
    kw = dict(maps=[m.to(device, dt).contiguous() for m in det_outputs], coeffs=pp._dummy_coeffs) if l1 else {}
    head = None if l1 else det_outputs.to(device, dt).contiguous()
    gt = det_boxes_gt.to(device).contiguous().float() if det_boxes_gt is not None else None
    pp.run(head, pp._dummy_protos, gt, pp._dummy_masks, pp._dummy_w, 0.0, stage="decode_filter", **kw)
    pp.run(head, pp._dummy_protos, gt, pp._dummy_masks, pp._dummy_w, 0.0, stage="nms_match", **kw)
    return pp.to_reference_lists()


def postprocess_infer(out_dict, det_boxes_gt, masks_gt, proj_weight, proj_bias=0.0, *, img_size=640, nc=3, device=None,
                      **cfg_kw):
    """Whole hot path on what ``model(imgs, mode="infer")`` returns (`main_modelv2.py:362-378`; SURVEY.md §7 item 2).

    ``out_dict["segment_preds_cat"]`` is the L2 head ``[B, 4+nc+32, N]``, ``out_dict["segment_protos"]`` the prototype
    tensor or the nested tuple the Ultralytics eval forward returns (unpacked with the reference's checks,
    `evaluate_model.py:142-159`).  ``masks_gt`` is ``[B,1,S,S]`` uint8 (or the dataset's float32 0/1,
    `dataset_btxrdv2.py:164-166`), ``proj_weight`` / ``proj_bias`` the `seg_proto_projector` parameters.  Returns
    ``(outputs, processor)``: the padded device tensors of ``PostProcessor.run`` and the processor (for
    ``to_reference_lists()``).  Extra keyword arguments go to ``PostConfig``."""
    head, protos = unpack_infer_dict(out_dict, nc=nc, proto_ch=32)
    device = torch.device(device) if device is not None else head.device
    B = head.shape[0]
    f32mask = masks_gt.dtype == torch.float32
    key = ("infer", B, img_size, nc, head.dtype, protos.dtype, f32mask, str(device), CONF_TH, NMS_IOU, TOP_K,
           tuple(sorted((k, str(v)) for k, v in cfg_kw.items())))
    pp = _cached.get(key)
    if pp is None:
        cfg = PostConfig(batch=B, img_size=img_size, nc=nc, head_bf16=head.dtype == torch.bfloat16,
                         proto_bf16=protos.dtype == torch.bfloat16, num_anchors=head.shape[2],
                         gt_mask_dtype=_lib.MASK_F32 if f32mask else _lib.MASK_U8, **cfg_kw)
        pp = _cached[key] = PostProcessor(cfg, device)
    gt = det_boxes_gt.to(device).contiguous().float() if det_boxes_gt is not None else None
    w = proj_weight.to(device).reshape(-1).contiguous().float()
    out = pp.run(head.to(device).contiguous(), protos.to(device).contiguous(), gt, masks_gt.to(device).contiguous(), w,
                 float(proj_bias))
    return out, pp
