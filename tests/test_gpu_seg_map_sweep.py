"""-m gpu: the v3 segmentation mAP from the records the mask stage appends (BtIO.seg_sweep, DeviceSweep(seg_map_capacity))
against the host path (btpost.segmap on the same outputs) and the oracle's COCO accumulate, through PostProcessor and
through Pipeline's captured steps."""
import numpy as np
import pytest
import torch

import helpers
from btpost import Pipeline, PostConfig, PostProcessor, _lib
from btpost.segmap import seg_map_outputs
from btpost.sweep import DeviceSweep, decode_records
from oracle import oracle

pytestmark = pytest.mark.gpu

THRS = oracle.iou_thresholds()
MAX_DETS = (1, 10, 100)


def seg_batch(B, S, seed, image_offset=0):
    """A synthetic batch whose projector mask follows the GT mask (the synthetic projector scores 0.0 seg mAP):
    proj_weight = e0 and prototype channel 0 = +c / -c from the GT mask sampled at the prototype pixel centres, with c
    varying per image.  Every fourth image gets an all-negative channel (empty mask: score exactly 0, tied across
    images), every fourth a channel shifted by a few prototype pixels (IoU spread over about 0.55 .. 0.95)."""
    batch = helpers.make(batch=B, img_size=S, seed=seed, image_offset=image_offset)
    PH, k = S // 4, S // 160
    centres = 4 * np.arange(PH) + 2
    samp = batch["masks_gt"][:, 0][:, centres][:, :, centres] > 0
    protos = batch["protos"].copy()
    for b in range(B):
        g = image_offset + b
        amp = np.float32(0.25 + 0.37 * ((g * 7 + 3) % 11))
        s = samp[b]
        if g % 4 == 2:
            s = np.zeros_like(s)
        elif g % 4 == 3:
            s = np.roll(s, (k * (1 + g % 3), k * (g % 2)), (0, 1))
        protos[b, 0] = np.where(s, amp, -amp)
    batch["protos"] = protos
    batch["proj_weight"] = np.eye(32, dtype=np.float32)[0]
    batch["proj_bias"] = np.float32(0.0)
    return batch


def cfg_for(B, S, **kw):
    return PostConfig(batch=B, img_size=S, max_det=20, gt_mode=1, with_coco=True, with_seg_map=True, **kw)


def run(pp, batch, offset):
    d = helpers.to_dev(batch, "cuda:0")
    out = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"], image_offset=offset)
    torch.cuda.synchronize()
    return out


def oracle_seg_ap(img3, scores):
    """oracle.accumulate_ap (nc = 1) over oracle.seg_map_records of per-image (inter, |P|, |G|) and scores in global
    image order."""
    rec = oracle.seg_map_records(img3, scores, THRS)
    recs = [dict(labels=np.zeros(1, np.int64), scores=rec["dets"][b, :1, 4], matched=rec["dt_match"][b] > 0,
                 ignored=rec["dt_ignore"][b] > 0) for b in range(len(scores))]
    npig = (1 - rec["gt_ignore"][:, :, 0].astype(np.int64)).sum(0)[:, None]
    return oracle.accumulate_ap(recs, npig, THRS, MAX_DETS, 1), npig


def assert_seg_tables(res, want):
    np.testing.assert_array_equal(res["seg_map_precision"], want["precision"])    # float64, bit for bit
    np.testing.assert_array_equal(res["seg_map_recall"], want["recall"])
    for k in ("map", "map_50", "map_75", "map_small", "map_medium", "map_large", "mar_1", "mar_10", "mar_100"):
        assert res[f"seg_{k}"] == want[k], k


@pytest.mark.parametrize("S", [160, 640])
def test_records_equal_host_prep_and_tables_equal_oracle(S):
    B, nb = 8, 2
    sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=B * nb * 20, max_det_per_image=20, device="cuda:0", seg_map_capacity=B * nb)
    pp = PostProcessor(cfg_for(B, S), "cuda:0", sweep=sweep)
    img3, scores = [], []
    for i in (1, 0):                                                 # batches out of order
        batch = seg_batch(B, S, 57 + S, image_offset=B * i)
        out = run(pp, batch, B * i)
        ref = oracle.run_pipeline(batch, img_size=S, max_det=20, gt_mode=1, with_instances=False, with_masks_out=False)
        np.testing.assert_array_equal(out["seg_img3"].cpu().numpy(), ref["seg_img3"])
        host = seg_map_outputs(pp.out, THRS)                         # the host path on the same step's outputs
        n = int(sweep.seg_hdr[_lib.SWEEP_N_RECORDS])
        rec = decode_records(sweep.seg_records[:n], len(THRS))
        sel = np.nonzero((rec["image"] >= B * i) & (rec["image"] < B * i + B))[0]
        sel = sel[np.argsort(rec["image"][sel])]
        np.testing.assert_array_equal(rec["image"][sel], B * i + np.arange(B))
        assert rec["score"][sel].tobytes() == host["seg_map_score"].cpu().numpy().tobytes()
        np.testing.assert_array_equal(rec["matched"][sel], host["dt_match"].cpu().numpy()[..., 0] > 0)
        np.testing.assert_array_equal(rec["ignored"][sel], host["dt_ignore"].cpu().numpy()[..., 0] > 0)
        assert not (rec["label"][sel].any() or rec["rank"][sel].any() or rec["class_rank"][sel].any())
        img3.insert(0, out["seg_img3"].cpu().numpy().copy()); scores.insert(0, host["seg_map_score"].cpu().numpy().copy())
    img3, scores = np.concatenate(img3), np.concatenate(scores)
    assert (scores == 0).sum() >= 2                                  # ties across images
    want, npig = oracle_seg_ap(img3, scores)
    h = sweep.seg_hdr.cpu().numpy()
    assert h[_lib.SWEEP_N_IMAGES] == B * nb and h[_lib.SWEEP_N_RECORDS] == B * nb
    np.testing.assert_array_equal(h[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64].reshape(4, 16)[:, :1], npig)
    assert not h[_lib.SWEEP_FSUM: _lib.SWEEP_FSUM + 4].any()
    res = sweep.finish()
    assert_seg_tables(res, want)
    assert 0.0 < res["seg_map_50"] < 1.0 and res["n_seg_records"] == B * nb


def test_pipeline_offsets_and_detection_results_unchanged():
    """Captured steps write the records (explicit offsets in scrambled order and auto_image_offset give the same seg
    tables), and the detection keys of finish() equal those of a sweep without a segmentation ring."""
    B, S, depth, nb = 4, 160, 3, 6
    batches = {i: seg_batch(B, S, 91, image_offset=B * i) for i in range(nb)}
    w = helpers.to_dev(batches[0], "cuda:0")["proj_weight"]
    results = {}
    for mode in ("scrambled", "auto", "no_seg"):
        seg = mode != "no_seg"
        sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=nb * B * 20, max_det_per_image=20, device="cuda:0",
                            seg_map_capacity=nb * B if seg else 0)
        pipe = Pipeline(cfg_for(B, S) if seg else PostConfig(batch=B, img_size=S, max_det=20, gt_mode=1, with_coco=True),
                        "cuda:0", depth=depth, proj_weight=w, sweep=sweep, auto_image_offset=mode == "auto")
        for i in ((3, 0, 5, 1, 4, 2) if mode == "scrambled" else range(nb)):
            d = helpers.to_dev(batches[i], "cuda:0")
            pipe.submit(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], image_offset=None if mode == "auto" else B * i)
        pipe.join()
        torch.cuda.synchronize()
        results[mode] = sweep.finish()
    a, b, base = results["scrambled"], results["auto"], results["no_seg"]
    for k in ("seg_map_precision", "seg_map_recall"):
        np.testing.assert_array_equal(a[k], b[k])
    assert a["n_seg_records"] == b["n_seg_records"] == nb * B and 0.0 < a["seg_map_50"] < 1.0
    for r in (a, b):
        for k, v in base.items():
            if isinstance(v, (np.ndarray, torch.Tensor)):
                np.testing.assert_array_equal(np.asarray(r[k]), np.asarray(v), err_msg=k)
            else:
                assert r[k] == v, k
    # the oracle's accumulate over the (inter, |P|, |G|) and scores of the same images, one PostProcessor step per batch
    pp = PostProcessor(cfg_for(B, S), "cuda:0")
    img3, scores = [], []
    for i in range(nb):
        out = run(pp, batches[i], B * i)
        img3.append(out["seg_img3"].cpu().numpy().copy())
        scores.append(seg_map_outputs(out, THRS)["seg_map_score"].cpu().numpy().copy())
    want, _ = oracle_seg_ap(np.concatenate(img3), np.concatenate(scores))
    assert_seg_tables(a, want)


def test_seg_ring_overflow_and_config_check():
    B, S = 4, 160
    small = DeviceSweep(3, THRS, MAX_DETS, capacity=4096, max_det_per_image=20, device="cuda:0", seg_map_capacity=3)
    pp = PostProcessor(cfg_for(B, S), "cuda:0", sweep=small)
    run(pp, seg_batch(B, S, 5), 0)
    assert int(small.seg_hdr[_lib.SWEEP_N_RECORDS]) == B
    with pytest.raises(RuntimeError, match="ring too small"):
        small.finish()
    with pytest.raises(ValueError, match="with_seg_map"):
        PostProcessor(PostConfig(batch=B, img_size=S, max_det=20, with_coco=True), "cuda:0", sweep=small)
