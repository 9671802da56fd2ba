"""-m gpu: binned PR / ROC curves of the projector probabilities (btpost_seg_curve, PostConfig.seg_curve,
DeviceSweep(seg_curve=...)) against the numpy restatement of tests/seg_curve_oracle.py on the oracle's upsampled logits:
hist bit for bit, every other output byte for byte unchanged, and the sweep's AP / AUROC exactly."""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers
import seg_curve_oracle as sco
from btpost import Pipeline, PostConfig, PostProcessor, _lib, segcurve
from btpost.sweep import DeviceSweep
from oracle import oracle
from test_gpu_soft_dice import soft_batch

pytestmark = pytest.mark.gpu

THRS = oracle.iou_thresholds()
MAX_DETS = (1, 10, 100)
HALF_DN, HALF_UP = np.nextafter(np.float32(0.5), np.float32(0)), np.nextafter(np.float32(0.5), np.float32(1))
THRESHOLD_SPECS = {"T2": 2, "T101": 101, "T1024": 1024, "hand": [0.0, float(HALF_DN), 0.5, float(HALF_UP), 1.0]}


def cfg_for(B, S, **kw):
    return PostConfig(batch=B, img_size=S, max_det=20, gt_mode=1, with_coco=True, **kw)


def run(pp, batch, bias=None):
    d = helpers.to_dev(batch, "cuda:0", gt_f32=pp.cfg.gt_mask_dtype == _lib.MASK_F32, proto_bf16=pp.cfg.proto_bf16)
    out = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"],
                 d["proj_bias"] if bias is None else bias)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def curve(pp, thr):
    """btpost_seg_curve on what pp's last run left in its workspace, into a fresh hist; returns it (numpy)."""
    thr = np.asarray(thr, np.float32)
    hist = torch.zeros(2, len(thr) + 1, dtype=torch.int64, device="cuda:0")
    rc = pp.lib.btpost_seg_curve(C.byref(pp.params), C.c_void_p(pp._ws_ptr), C.c_size_t(pp._ws_bytes),
                                 (C.c_float * len(thr))(*thr.tolist()), len(thr), C.c_void_p(hist.data_ptr()),
                                 C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "btpost_seg_curve")
    torch.cuda.synchronize()
    return hist.cpu().numpy()


def oracle_logits(batch, S, proto_bf16=False, bias=None):
    protos = batch["protos"]
    if proto_bf16:   # the kernels widen the bf16 prototypes exactly: the oracle sees the same values
        protos = torch.from_numpy(protos).bfloat16().float().numpy()
    b0 = batch["proj_bias"] if bias is None else np.float32(bias)
    return np.stack([oracle.project_upsample(protos[b], batch["proj_weight"], b0, S)[1] for b in range(protos.shape[0])])


def curve_batch(B, S, seed):
    """The synthetic batch (its projector's logits spread over the whole sigmoid) with image 1's logits scaled up to
    +-hundreds, so that p = 0 (x < -87) and p = 1 occur."""
    batch = helpers.make(batch=B, img_size=S, seed=seed)
    batch["protos"][1] *= np.float32(120.0)
    return batch


@pytest.mark.parametrize("bf16,gt_f32", [(False, False), (True, True)], ids=["f32-u8", "bf16-f32gt"])
@pytest.mark.parametrize("S", [160, 640, 1024])
def test_hist_equals_restatement(S, bf16, gt_f32):
    B = 3 if S == 1024 else 4
    batch = curve_batch(B, S, 700 + S + bf16)
    pp = PostProcessor(cfg_for(B, S, proto_bf16=bf16, gt_mask_dtype=_lib.MASK_F32 if gt_f32 else _lib.MASK_U8), "cuda:0")
    out = run(pp, batch)
    up = oracle_logits(batch, S, bf16)
    gt = batch["masks_gt"][:, 0]
    for name, spec in THRESHOLD_SPECS.items():
        thr = segcurve.thresholds(spec)
        got = curve(pp, thr)
        np.testing.assert_array_equal(got, sco.seg_curve_hist(up, gt, thr), err_msg=name)
        assert got.sum() == B * S * S and got[1].sum() == out["seg_img3"][:, 2].sum()
        assert got[:, 1:-1].any()                                   # probabilities between the outer thresholds
        np.testing.assert_array_equal(curve(pp, thr), got)         # a repeated call writes the same words


def test_constant_probability_pins_greater_equal():
    """proj_weight = 0 and a short-mantissa bias: every logit is the bias exactly, every pixel has one known p.  A
    threshold at p counts it as positive, the next fp32 value above p does not."""
    B, S, bias = 2, 160, 0.375
    batch = helpers.make(batch=B, img_size=S, seed=5)
    batch["proj_weight"] = np.zeros(32, np.float32)
    pp = PostProcessor(cfg_for(B, S), "cuda:0")
    out = run(pp, batch, bias)
    p = sco.soft_prob(np.float32([bias]))[0]
    below, above = np.nextafter(p, np.float32(0)), np.nextafter(p, np.float32(1))
    n, g = B * S * S, int(out["seg_img3"][:, 2].sum())
    for thr, j in (([below, p, above], 2), ([0.0, below], 2), ([p, p], 2), ([above, 1.0], 0), ([below, above], 1)):
        got = curve(pp, thr)
        want = np.zeros_like(got)
        want[0, j], want[1, j] = n - g, g
        np.testing.assert_array_equal(got, want, err_msg=str(thr))


def test_threshold_half_against_seg_cnt4():
    """At the fp32 threshold 0.5 the curve (p >= 0.5) and the mask stage's `sigmoid(x) > 0.5` disagree only on pixels
    with |x| < 2^-20 (checked through seg_logits)."""
    B, S = 4, 640
    batch = helpers.make(batch=B, img_size=S, seed=31)
    pp = PostProcessor(cfg_for(B, S, with_seg_logits=True, with_seg_mask=True), "cuda:0")
    out = run(pp, batch)
    h = curve(pp, [0.0, 0.5])
    x, mask, gt = out["seg_logits"], out["seg_mask"] != 0, batch["masks_gt"][:, 0] != 0
    pos = sco.soft_prob(x) >= np.float32(0.5)
    assert (np.abs(x[pos != mask]) < 2.0 ** -20).all()
    tp, fp = int(h[1, 2]), int(h[0, 2])
    cnt4 = out["seg_cnt4"]
    assert tp - int(cnt4[0]) == int((pos & ~mask & gt).sum()) - int((~pos & mask & gt).sum())
    assert fp - int(cnt4[1]) == int((pos & ~mask & ~gt).sum()) - int((~pos & mask & ~gt).sum())


VARIANTS = {"alone": {}, "soft_dice": dict(with_soft_dice=True), "seg_map": dict(with_seg_map=True),
            "surface": dict(with_surface_dist=True),
            "all": dict(with_soft_dice=True, with_seg_map=True, with_surface_dist=True, with_seg_logits=True)}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_other_outputs_unchanged(variant):
    B, S = 4, 160
    batch = soft_batch(B, S, 820)
    got = run(PostProcessor(cfg_for(B, S, seg_curve=101, **VARIANTS[variant]), "cuda:0"), batch)
    base = run(PostProcessor(cfg_for(B, S, **VARIANTS[variant]), "cuda:0"), batch)
    thr = segcurve.thresholds(101)
    np.testing.assert_array_equal(got["seg_curve"], sco.seg_curve_hist(oracle_logits(batch, S), batch["masks_gt"][:, 0], thr))
    assert set(got) == set(base) | {"seg_curve"}
    for k, v in base.items():
        assert got[k].tobytes() == v.tobytes(), k                  # bit for bit, floats too


def test_single_images_sum_to_the_batch():
    B, S = 5, 160
    batch = curve_batch(B, S, 44)
    whole = run(PostProcessor(cfg_for(B, S, seg_curve=101), "cuda:0"), batch)["seg_curve"]
    pp1 = PostProcessor(cfg_for(1, S, seg_curve=101), "cuda:0")
    for b in range(B):
        one = {k: (v[b: b + 1] if isinstance(v, np.ndarray) and v.ndim and v.shape[0] == B and k != "det_boxes_gt" else v)
               for k, v in batch.items()}
        rows = batch["det_boxes_gt"][batch["det_boxes_gt"][:, 0] == b].copy()
        rows[:, 0] = 0
        one["det_boxes_gt"] = rows
        run(pp1, one)
    np.testing.assert_array_equal(pp1.out["seg_curve"].cpu().numpy(), whole)   # accumulated over the five calls


def test_pipeline_and_device_sweep():
    """Captured Pipeline steps (depths 2 and 3, auto_image_offset) give the serial calls' words; finish() returns the
    restatement's AP / AUROC exactly."""
    B, S, nb = 4, 160, 5
    batches = [curve_batch(B, S, 60 + i) for i in range(nb)]
    for bt in batches[1:]:                                         # a Pipeline holds one projector
        bt["proj_weight"], bt["proj_bias"] = batches[0]["proj_weight"], batches[0]["proj_bias"]
    thr = segcurve.thresholds(101)
    want = sum(sco.seg_curve_hist(oracle_logits(b, S), b["masks_gt"][:, 0], thr) for b in batches)
    serial = PostProcessor(cfg_for(B, S, seg_curve=101), "cuda:0")
    for b in batches:
        run(serial, b)
    np.testing.assert_array_equal(serial.out["seg_curve"].cpu().numpy(), want)
    m = segcurve.curve_metrics(segcurve.confmat(want), thr)
    w = helpers.to_dev(batches[0], "cuda:0")["proj_weight"]
    for depth, use_sweep in ((2, True), (3, True), (2, False)):
        sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=nb * B * 20, max_det_per_image=20, device="cuda:0",
                            seg_curve=101) if use_sweep else None
        pipe = Pipeline(cfg_for(B, S, seg_curve=101), "cuda:0", depth=depth, proj_weight=w,
                        proj_bias=float(batches[0]["proj_bias"]), sweep=sweep, auto_image_offset=True)
        for b in batches:
            d = helpers.to_dev(b, "cuda:0")
            pipe.submit(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"])
        pipe.join()
        torch.cuda.synchronize()
        np.testing.assert_array_equal(pipe.counters("seg_curve").cpu().numpy(), want, err_msg=str((depth, use_sweep)))
        if use_sweep:
            res = sweep.finish()
            assert res["seg_ap"] == m["ap"] and res["seg_auroc"] == m["auroc"] and res["n_images"] == nb * B
            np.testing.assert_array_equal(res["seg_curve_confmat"], segcurve.confmat(want))
            np.testing.assert_array_equal(res["seg_curve_thresholds"], thr)
            for key, mk in (("seg_pr_curve", "pr_curve"), ("seg_roc", "roc")):
                for a, b in zip(res[key], m[mk]):
                    np.testing.assert_array_equal(a, b)
            sweep.reset()
            assert not sweep.seg_curve.any()


def test_config_mismatch_raises():
    sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=4096, max_det_per_image=20, device="cuda:0", seg_curve=101)
    with pytest.raises(ValueError, match="seg_curve"):
        PostProcessor(cfg_for(4, 160), "cuda:0", sweep=sweep)
    with pytest.raises(ValueError, match="differ"):
        PostProcessor(cfg_for(4, 160, seg_curve=100), "cuda:0", sweep=sweep)
    with pytest.raises(ValueError, match="seg_curve"):
        PostProcessor(cfg_for(4, 160, seg_curve=101), "cuda:0",
                      sweep=DeviceSweep(3, THRS, MAX_DETS, capacity=4096, max_det_per_image=20, device="cuda:0"))
    PostProcessor(cfg_for(4, 160, seg_curve=list(segcurve.thresholds(101))), "cuda:0", sweep=sweep)
    res = sweep.finish()
    assert not res["seg_curve_confmat"].any() and res["seg_ap"] == 0.0
