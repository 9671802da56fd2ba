"""Shared test helpers: run the CUDA library and the CPU oracle on the same synthetic batch."""
import numpy as np
import torch

from btpost import PostConfig, PostProcessor, _lib, synth
from oracle import oracle


def to_dev(batch, dev, gt_f32=False, proto_bf16=False, head_bf16=False):
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    m = batch["masks_gt"].astype(np.float32) if gt_f32 else batch["masks_gt"]
    protos = t(batch["protos"]).bfloat16() if proto_bf16 else t(batch["protos"])
    head = t(batch["head"]).bfloat16() if head_bf16 else t(batch["head"])
    return dict(head=head, protos=protos, det_boxes_gt=t(batch["det_boxes_gt"]),
                masks_gt=t(m), proj_weight=t(batch["proj_weight"]), proj_bias=float(batch["proj_bias"]))


def run_cuda(batch, dev="cuda:0", gt_f32=False, l1=False, **kw):
    scfg = batch["cfg"]
    cfg = PostConfig(batch=scfg.batch, img_size=scfg.img_size, nc=scfg.nc, nm=scfg.nm,
                     layout=_lib.LAYOUT_L1 if l1 else _lib.LAYOUT_L2,
                     conf_thres=kw.get("conf_thres", 0.05), iou_thres=kw.get("iou_thres", 0.6),
                     max_det=kw.get("max_det", 300), max_cand=kw.get("max_cand", 0),
                     class_mode=kw.get("class_mode", 0), clamp_boxes=bool(kw.get("clamp", 1)),
                     gt_mode=kw.get("gt_mode", 0), crop=bool(kw.get("crop", 1)),
                     iou_match_thresh=kw.get("iou_match_thresh", 0.5),
                     gt_mask_dtype=_lib.MASK_F32 if gt_f32 else _lib.MASK_U8, nms_threads=kw.get("nms_threads", 0),
                     proto_bf16=bool(kw.get("proto_bf16", False)), head_bf16=bool(kw.get("head_bf16", False)),
                     drop_gt_no_cand=bool(kw.get("drop_gt_no_cand", 0)), with_inst_masks=kw.get("with_inst_masks"),
                     num_anchors=kw.get("num_anchors"), with_seg_mask=True, with_seg_logits=True, with_uni_mask=True, with_coco=True, with_seg_map=True,
                     with_soft_dice=bool(kw.get("with_soft_dice", False)))
    pp = PostProcessor(cfg, dev)
    d = to_dev(batch, dev, gt_f32, bool(kw.get("proto_bf16", False)), bool(kw.get("head_bf16", False)))
    extra = {}
    if l1:
        cast = (lambda t: t.bfloat16()) if kw.get("head_bf16") else (lambda t: t)
        extra = dict(maps=[cast(torch.from_numpy(m).to(dev)) for m in batch["maps"]], coeffs=cast(torch.from_numpy(batch["coeffs"]).to(dev)))
    out = pp.run(None if l1 else d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"],
                 **extra)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}, pp


def make(batch=2, img_size=640, seed=20261, l1=False, image_offset=0, nc=3):
    cfg = synth.SynthConfig(batch=batch, img_size=img_size, seed=seed, image_offset=image_offset, nc=nc)
    b = synth.make_batch(cfg, l1=l1)
    b["cfg"] = cfg
    return b


def assert_same(got, ref, B, max_det, check_masks=True):
    """Bit-exact comparison of every output the oracle produces."""
    np.testing.assert_array_equal(got["n_cand"], ref["n_cand"])
    np.testing.assert_array_equal(got["det_count"], ref["det_count"])
    np.testing.assert_array_equal(got["det_keep"], ref["det_keep"].astype(np.int64))
    np.testing.assert_array_equal(got["det_anchor"], ref["det_anchor"])
    assert got["dets"].tobytes() == ref["dets"].tobytes()
    assert got["det_coeff"].tobytes() == ref["det_coeff"].tobytes()
    np.testing.assert_array_equal(got["gt_count"], ref["gt_count"])
    assert got["gt_boxes"].tobytes() == ref["gt_boxes"].tobytes()
    assert got["gt_boxes_raw"].tobytes() == ref["gt_boxes_raw"].tobytes()
    np.testing.assert_array_equal(got["gt_labels"], ref["gt_labels"])
    np.testing.assert_array_equal(got["cm"], ref["cm"])
    np.testing.assert_array_equal(got["cm_pos"], ref["cm_pos"])
    np.testing.assert_array_equal(got["seg_cnt4"], ref["seg_cnt4"])
    np.testing.assert_array_equal(got["seg_img3"], ref["seg_img3"])
    np.testing.assert_allclose(got["seg_dice"], ref["seg_dice"], rtol=1e-5)   # north star: 1e-5 relative on floats
    np.testing.assert_allclose(got["seg_iou"], ref["seg_iou"], rtol=1e-5)
    if check_masks:
        np.testing.assert_array_equal(got["seg_mask"], ref["seg_mask"])
        assert got["seg_logits"].tobytes() == ref["seg_logits"].tobytes()
    if ref["inst_masks"]:
        np.testing.assert_array_equal(got["inst_area"], ref["inst_area"])
        np.testing.assert_array_equal(got["inst_inter"], ref["inst_inter"])
        np.testing.assert_array_equal(got["uni_img3"], ref["uni_img3"])
        np.testing.assert_array_equal(got["uni_cnt4"], ref["uni_cnt4"])
        np.testing.assert_allclose(got["uni_dice"], ref["uni_dice"], rtol=1e-5)
        np.testing.assert_allclose(got["uni_iou"], ref["uni_iou"], rtol=1e-5)
        if check_masks:
            np.testing.assert_array_equal(got["uni_mask"], ref["uni_mask"])
        if "inst_bits" in got:   # every instance bitmap, pixel for pixel (src/test_model.py:80-85 + crop)
            for b in range(B):
                k = int(ref["det_count"][b])
                planes = np.unpackbits(got["inst_bits"][b], axis=-1, bitorder="little")
                np.testing.assert_array_equal(planes[:k], ref["inst_masks"][b], err_msg=f"instance masks of image {b}")
                assert not planes[k:].any(), "planes beyond det_count must be zero"
                if "inst_masks" in got:
                    np.testing.assert_array_equal(got["inst_masks"][b], planes)
    np.testing.assert_array_equal(got["dt_match"], ref["dt_match"])
    np.testing.assert_array_equal(got["dt_ignore"], ref["dt_ignore"])
    np.testing.assert_array_equal(got["gt_ignore"], ref["gt_ignore"])


def oracle_parallel(batch, workers=None, chunk=1, **kw):
    """oracle.run_pipeline over chunks of images on a thread pool (the C parts release the GIL); outputs are
    concatenated, the accumulated counters summed.  Same results as one call over the whole batch."""
    import os
    from concurrent.futures import ThreadPoolExecutor
    B = batch["protos"].shape[0]
    gt = batch["det_boxes_gt"]

    def one(b0):
        b1 = min(B, b0 + chunk)
        sub = dict(batch)
        for k in ("head", "protos", "masks_gt", "coeffs"):
            if k in batch:
                sub[k] = batch[k][b0:b1]
        if "maps" in batch:                        # the raw-map (L1) layout: three per-level maps
            sub["maps"] = [m[b0:b1] for m in batch["maps"]]
        rows = gt[(gt[:, 0] >= b0) & (gt[:, 0] < b1)].copy() if len(gt) else gt
        if len(rows):
            rows[:, 0] -= b0
        sub["det_boxes_gt"] = rows
        return oracle.run_pipeline(sub, **kw)

    with ThreadPoolExecutor(workers or os.cpu_count() or 4) as pool:
        parts = list(pool.map(one, range(0, B, chunk)))
    out = {}
    for k, v in parts[0].items():
        if k in ("cm", "seg_cnt4", "uni_cnt4"):
            out[k] = sum(p[k] for p in parts)
        elif isinstance(v, list):
            out[k] = [x for p in parts for x in p[k]]
        elif v is None:
            out[k] = None
        else:
            out[k] = np.concatenate([p[k] for p in parts], 0)
    return out
