"""-m gpu: v3's soft Dice on the projector probabilities (BtIOSoftDice.seg_soft2 / seg_soft_dice / seg_soft_acc,
PostConfig.with_soft_dice, DeviceSweep(soft_dice=True)) against the numpy restatement of tests/soft_dice_oracle.py on the
oracle's upsampled logits: the fixed-point sums bit for bit, the per-image value and the sweep's mean exactly."""
import numpy as np
import pytest
import torch

import helpers
import soft_dice_oracle as sd
from btpost import Pipeline, PostConfig, PostProcessor
from btpost.sweep import DeviceSweep
from oracle import oracle
from test_gpu_seg_map_sweep import seg_batch

pytestmark = pytest.mark.gpu

THRS = oracle.iou_thresholds()
MAX_DETS = (1, 10, 100)
SOFT_KEYS = ("seg_soft2", "seg_soft_dice", "seg_soft_acc")


def soft_batch(B, S, seed, image_offset=0):
    """seg_batch (a projector that follows the GT mask, empty and shifted masks among the images) with the logits of
    its second image scaled up to +-hundreds, so that both ends of the sigmoid (p = 0 below -87, p = 1) occur."""
    batch = seg_batch(B, S, seed, image_offset)
    batch["protos"][1, 0] *= np.float32(120.0)
    return batch


def oracle_soft(batch, S, proto_bf16=False, bias=None):
    """(seg_soft2 [B, 2], seg_soft_dice [B]) of the restatement on the oracle's upsampled projector logits."""
    protos = batch["protos"]
    if proto_bf16:   # the kernels widen the bf16 prototypes exactly: the oracle sees the same values
        protos = torch.from_numpy(protos).bfloat16().float().numpy()
    b0 = batch["proj_bias"] if bias is None else np.float32(bias)
    up = np.stack([oracle.project_upsample(protos[b], batch["proj_weight"], b0, S)[1] for b in range(protos.shape[0])])
    gt = batch["masks_gt"][:, 0] != 0
    soft2 = sd.soft_sums(up, gt)
    return soft2, sd.soft_dice(soft2, gt.reshape(len(gt), -1).sum(1))


def cfg_for(B, S, **kw):
    return PostConfig(batch=B, img_size=S, max_det=20, gt_mode=1, with_coco=True, **kw)


def run(pp, batch, bias=None):
    d = helpers.to_dev(batch, "cuda:0", proto_bf16=pp.cfg.proto_bf16)
    out = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"],
                 d["proj_bias"] if bias is None else bias)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


# every branch of m1_item's dense path: soft Dice alone, with the v3 seg-mAP score, with the dense outputs, with all
VARIANTS = {"alone": {}, "seg_map": dict(with_seg_map=True), "dense": dict(with_seg_logits=True, with_seg_mask=True),
            "all": dict(with_seg_map=True, with_seg_logits=True, with_seg_mask=True)}


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("S", [160, 640])
def test_soft_dice_equals_oracle_and_leaves_other_outputs_unchanged(S, bf16, variant):
    B = 4 if S == 160 else 3
    batch = soft_batch(B, S, 300 + S + bf16)
    kw = dict(VARIANTS[variant], proto_bf16=bf16)
    got = run(PostProcessor(cfg_for(B, S, with_soft_dice=True, **kw), "cuda:0"), batch)
    base = run(PostProcessor(cfg_for(B, S, **kw), "cuda:0"), batch)
    soft2, dice = oracle_soft(batch, S, bf16)
    np.testing.assert_array_equal(got["seg_soft2"], soft2)
    np.testing.assert_array_equal(got["seg_soft_dice"], dice)                    # fp32, NaN where undefined
    np.testing.assert_array_equal(got["seg_soft_acc"], sd.accumulate(dice))
    assert np.isfinite(dice).all() and 0.0 < dice.min() and dice.max() < 1.0   # every image has GT pixels here
    assert set(got) == set(base) | set(SOFT_KEYS)
    for k, v in base.items():
        assert got[k].tobytes() == v.tobytes(), k                              # bit for bit, floats too


def test_pipeline_and_device_sweep():
    """Captured Pipeline steps (auto_image_offset) add every image into the sweep's seg_soft_acc: finish() returns the
    restatement's mean over the same images, and the accumulator words do not depend on the pipeline depth (nor on
    whether they live in a sweep header or in Pipeline.shared)."""
    B, S, nb = 4, 160, 6
    batches = [soft_batch(B, S, 77, image_offset=B * i) for i in range(nb)]
    want = sd.accumulate(np.concatenate([oracle_soft(b, S)[1] for b in batches]))
    w = helpers.to_dev(batches[0], "cuda:0")["proj_weight"]
    words = {}
    for depth, use_sweep in ((2, True), (3, True), (2, False)):
        sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=nb * B * 20, max_det_per_image=20, device="cuda:0",
                            soft_dice=True) if use_sweep else None
        pipe = Pipeline(cfg_for(B, S, with_soft_dice=True), "cuda:0", depth=depth, proj_weight=w, sweep=sweep,
                        auto_image_offset=True)
        for b in batches:
            d = helpers.to_dev(b, "cuda:0")
            pipe.submit(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"])
        pipe.join()
        torch.cuda.synchronize()
        words[(depth, use_sweep)] = pipe.counters("seg_soft_acc").cpu().numpy().copy()
        if use_sweep:
            res = sweep.finish()
            assert res["n_soft_dice_images"] == nb * B and res["n_images"] == nb * B
            assert res["seg_soft_dice"] == sd.mean(want)
    for v in words.values():
        np.testing.assert_array_equal(v, want)


def test_undefined_soft_dice_is_nan_and_not_counted():
    """A projector bias that drives every logit below -87 gives p = 0 everywhere: an image with an empty GT mask has
    P + G == 0, its soft Dice is NaN and the accumulator leaves it out; the others score exactly 0."""
    B, S, bias = 3, 160, -200.0
    batch = seg_batch(B, S, 11)
    batch["masks_gt"][0] = 0
    assert (batch["masks_gt"][1:].reshape(B - 1, -1) != 0).any(1).all()
    sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=4096, max_det_per_image=20, device="cuda:0", soft_dice=True)
    pp = PostProcessor(cfg_for(B, S, with_soft_dice=True), "cuda:0", sweep=sweep)
    out = run(pp, batch, bias)
    soft2, dice = oracle_soft(batch, S, bias=bias)
    assert not soft2.any() and np.isnan(dice[0]) and (dice[1:] == 0).all()
    np.testing.assert_array_equal(out["seg_soft2"], soft2)
    np.testing.assert_array_equal(out["seg_soft_dice"], dice)
    res = sweep.finish()
    assert res["n_soft_dice_images"] == B - 1 and res["seg_soft_dice"] == 0.0
    # no image with a defined value: the mean is NaN
    sweep.reset()
    batch["masks_gt"][:] = 0
    run(pp, batch, bias)
    res = sweep.finish()
    assert res["n_soft_dice_images"] == 0 and np.isnan(res["seg_soft_dice"])


def test_soft_dice_sweep_needs_with_soft_dice():
    sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=4096, max_det_per_image=20, device="cuda:0", soft_dice=True)
    with pytest.raises(ValueError, match="with_soft_dice"):
        PostProcessor(cfg_for(4, 160), "cuda:0", sweep=sweep)
    PostProcessor(cfg_for(4, 160, with_soft_dice=True), "cuda:0", sweep=sweep)
