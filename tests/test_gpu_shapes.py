"""-m gpu: the shapes, class counts and dtypes that select the decode kernel's variants and the mask stage's tile
remainders the other GPU tests never reach.  Each case is named after the variant it selects (`l2-f32-vec1-320` is
decode_filter_l2_kernel<VEC = 1, MAXT = 320> on an fp32 head; `pw24` a prototype width whose last 32-column tile is
24 columns wide; see test_anchor_limits.py for the selection rule).  Every output is compared bit for bit with the
oracle, and the detections, projector logits and masks, Dice / IoU, soft Dice and instance masks with the float64
restatement of tests/f64_reference.py, which does not share the oracle's code."""
import numpy as np
import pytest
import torch

import f64_reference as f64
import helpers
from oracle import oracle

pytestmark = pytest.mark.gpu

SEED = 20286
# id, layout, bf16 inputs, image size, batch, classes
CASES = [
    ("l2-f32-vec1-320-tinytile", "l2", False, 32, 3, 3),     # 21 anchors over 8 CTAs (ranks without anchors); PW = 8
    ("l2-f32-vec1-320-pw24", "l2", False, 96, 2, 1),
    ("l2-f32-vec4-288-pw16", "l2", False, 320, 5, 16),
    ("l2-f32-vec1-1024-pw24", "l2", False, 480, 2, 2),
    ("l2-f32-vec4-320-pw16", "l2", False, 704, 1, 3),
    ("l2-bf16-vec1-320", "l2", True, 96, 2, 3),
    ("l2-bf16-vec1-1024", "l2", True, 480, 2, 3),
    ("l2-bf16-vec4-1024", "l2", True, 768, 2, 3),
    ("l1-f32-vec2-1024", "l1", False, 736, 1, 3),
    ("l1-f32-vec4-1024", "l1", False, 1024, 2, 3),
    ("l1-bf16-vec2-1024", "l1", True, 800, 1, 3),
    ("l1-bf16-vec4-1024", "l1", True, 960, 2, 3),
]
INST_MAX_S = 480        # above it the oracle's instance masks cost minutes: they are compared up to 480^2


def _bf16(a):
    return torch.from_numpy(np.ascontiguousarray(a)).bfloat16().float().numpy()


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_variant_matches_oracle_and_float64_reference(case):
    name, layout, bf16, S, B, nc = case
    l1 = layout == "l1"
    batch = helpers.make(batch=B, img_size=S, seed=SEED, l1=l1, nc=nc)
    if bf16:                                  # the kernels widen bf16 exactly: both references take the rounded tensors
        if l1:
            batch["maps"] = [_bf16(m) for m in batch["maps"]]
            batch["coeffs"] = _bf16(batch["coeffs"])
        else:
            batch["head"], batch["protos"] = _bf16(batch["head"]), _bf16(batch["protos"])
    inst = S <= INST_MAX_S
    gt_img = np.bincount(batch["det_boxes_gt"][:, 0].astype(np.int64), minlength=B)
    assert gt_img.min() > 0 and batch["masks_gt"].reshape(B, -1).sum(1).min() > 0
    for class_mode in ((0, 1, 2) if nc == 16 else (0,)):
        kw = dict(max_det=300, class_mode=class_mode)
        okw = dict(kw, img_size=S, nc=nc, with_instances=inst, **({"layout": "l1"} if l1 else {}))
        ref = helpers.oracle_parallel(batch, **okw)
        got, _ = helpers.run_cuda(batch, l1=l1, head_bf16=bf16, proto_bf16=bf16 and not l1, with_soft_dice=True,
                                  with_inst_masks="bits" if inst else None, **kw)
        assert got["det_count"].min() > 0 and got["gt_count"].min() > 0
        helpers.assert_same(got, ref, B, 300)
        if l1:
            labels = f64.check_l1_detections(batch["maps"], batch["coeffs"], got, nc, S)
        else:
            labels = f64.check_l2_detections(batch["head"], got, nc, S)
        if nc == 16:                          # the class loop, the 16 x 16 histogram and NPIG columns up to 15 ran
            assert labels.max() >= 8 and (got["gt_labels"][got["gt_count"][:, None] > np.arange(32)] >= 8).any()
            assert int(got["cm"][8:].sum() + got["cm"][:, 8:].sum()) > 0
        lg, E, n_band = f64.check_projector(batch["protos"], batch["proj_weight"], batch["proj_bias"], batch["masks_gt"],
                                            got, S)
        print(f"{name} class_mode {class_mode}: projector band {n_band} of {B * S * S} pixels")
        assert n_band <= 1e-3 * B * S * S
        f64.check_soft_dice(lg, E, batch["masks_gt"], got["seg_soft_dice"])
        if inst:
            planes = lambda b: np.unpackbits(got["inst_bits"][b], axis=-1, bitorder="little")[:int(got["det_count"][b])]
            n_inst = f64.check_instances(batch["protos"], got, planes, S)
            print(f"{name} class_mode {class_mode}: instance band {n_inst} of {int(got['det_count'].sum()) * S * S} pixels")
            assert n_inst <= 1e-3 * int(got["det_count"].sum()) * S * S


@pytest.mark.parametrize("nc", [1, 16])
def test_device_sweep_with_one_and_sixteen_classes(nc):
    """DeviceSweep fed by the library itself (records written by the COCO matching, NPIG[a][c] by class) with one class
    and with sixteen: finish()'s precision / recall tables and GT counts are bit-identical to the oracle's accumulate."""
    from btpost import PostConfig, PostProcessor
    from btpost.sweep import DeviceSweep, decode_records
    from test_gpu_sweep import _oracle_ap
    B, S = 4, 160
    kw = dict(max_det=100, gt_mode=1)
    sweep = DeviceSweep(nc, oracle.iou_thresholds(), (1, 10, 100), capacity=4096, max_det_per_image=100, device="cuda:0")
    pp = PostProcessor(PostConfig(batch=B, img_size=S, nc=nc, max_det=100, gt_mode=1, with_coco=True), "cuda:0", sweep=sweep)
    outs, offs = [], []
    for i in (2, 0, 1):
        batch = helpers.make(batch=B, img_size=S, seed=SEED, image_offset=B * i, nc=nc)
        ref = oracle.run_pipeline(batch, img_size=S, nc=nc, **kw)
        d = helpers.to_dev(batch, "cuda:0")
        out = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"], image_offset=B * i)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(out["dt_match"].cpu().numpy(), ref["dt_match"])
        outs.append(ref); offs.append(B * i)
    n = int(sweep.hdr[0])
    assert n == sum(int(o["det_count"].sum()) for o in outs)
    rec = decode_records(sweep.records[:n], 10)
    for ref, off in zip(outs, offs):
        for b in range(B):
            k = int(ref["det_count"][b])
            sel = np.nonzero(rec["image"] == off + b)[0]
            sel = sel[np.argsort(rec["rank"][sel])]
            lab = ref["dets"][b, :k, 5].astype(np.int64)
            np.testing.assert_array_equal(rec["label"][sel], lab)
            np.testing.assert_array_equal(rec["class_rank"][sel], [int((lab[:j] == lab[j]).sum()) for j in range(k)])
    want, npig = _oracle_ap(outs, offs, nc=nc)
    res = sweep.finish()
    assert res["n_images"] == 3 * B and res["n_records"] == n
    np.testing.assert_array_equal(res["npig"], npig)
    np.testing.assert_array_equal(res["precision"], want["precision"])      # float64, bit for bit
    np.testing.assert_array_equal(res["recall"], want["recall"])
    assert want["map_50"] > 0
    if nc == 16:
        assert npig[0, 8:].sum() > 0 and (rec["label"] >= 8).any()


def test_unsupported_anchor_count_and_misaligned_head_raise_early():
    """An L2 head of 672^2 (9261 anchors, N % 4 != 0, above the 8192 of the scalar decoder) is rejected when the
    processor is built, naming the anchor limit; a head that is not 16-byte aligned is rejected as misaligned instead of
    silently taking another decoder."""
    from btpost import PostConfig, PostProcessor
    with pytest.raises(ValueError, match="anchors"):
        PostProcessor(PostConfig(batch=1, img_size=672), "cuda:0")
    batch = helpers.make(batch=1, img_size=640, seed=SEED)
    d = helpers.to_dev(batch, "cuda:0")
    flat = torch.empty(d["head"].numel() + 1, dtype=torch.float32, device="cuda:0")
    head = flat[1:].view_as(d["head"])
    head.copy_(d["head"])
    assert head.is_contiguous() and head.data_ptr() % 16 == 4
    pp = PostProcessor(PostConfig(batch=1, img_size=640), "cuda:0")
    with pytest.raises(ValueError, match="misaligned"):
        pp.run(head, d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"])
