"""-m gpu: sweep aggregation on the device (the production placement) from the CUDA library's own outputs,
against the same aggregation on the CPU from the oracle's outputs."""
import numpy as np
import pytest
import torch

import helpers
from btpost import Pipeline, PostConfig, PostProcessor
from btpost.sweep import DeviceSweep, SweepState, decode_records
from oracle import oracle

pytestmark = pytest.mark.gpu


def test_device_sweep_matches_cpu_sweep_of_oracle_outputs():
    kw = dict(max_det=100, gt_mode=1)
    st_dev = SweepState(3, 10, oracle.iou_thresholds(), (1, 10, 100), device="cuda:0")
    st_cpu = SweepState(3, 10, oracle.iou_thresholds(), (1, 10, 100))
    pp = None
    for i in range(2):                                   # two batches of 4 images, 160^2
        batch = helpers.make(batch=4, img_size=160, seed=31, image_offset=4 * i)
        ref = oracle.run_pipeline(batch, img_size=160, **kw)
        got, pp_i = helpers.run_cuda(batch, **kw)
        helpers.assert_same(got, ref, 4, 100)
        st_dev.add(pp_i.out, 4 * i, accumulate_counters=True)
        st_cpu.add({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in ref.items() if isinstance(v, np.ndarray)}, 4 * i,
                   accumulate_counters=True)
    a, b = st_dev.compute(), st_cpu.compute()
    assert a["n_images"] == b["n_images"] == 8
    for k in ("map", "map_50", "map_75", "mar_1", "mar_10", "mar_100", "seg_f1", "seg_dice", "seg_iou", "uni_dice", "uni_iou"):
        assert float(a[k]) == pytest.approx(float(b[k]), rel=1e-6, abs=1e-9), k
    np.testing.assert_array_equal(a["cm"].cpu().numpy(), b["cm"].numpy())
    np.testing.assert_allclose(a["precision"].cpu().numpy(), b["precision"].numpy(), rtol=1e-12)


def _oracle_ap(outs, offsets, max_dets=(1, 10, 100), drop=False, nc=3):
    """oracle.accumulate_ap over a list of oracle batch outputs (images in global order)."""
    thrs = oracle.iou_thresholds()
    recs, npig = [], np.zeros((4, nc), np.int64)
    order = np.argsort(offsets)
    for i in order:
        out = outs[i]
        for b in range(len(out["det_count"])):
            k, g = int(out["det_count"][b]), int(out["gt_count"][b])
            recs.append(dict(labels=out["dets"][b, :k, 5].astype(np.int64), scores=out["dets"][b, :k, 4],
                             matched=out["dt_match"][b][:, :, :k] > 0, ignored=out["dt_ignore"][b][:, :, :k] > 0))
            if drop and int(out["n_cand"][b]) == 0:
                continue
            for a in range(4):
                for gi in range(g):
                    if not out["gt_ignore"][b, a, gi]:
                        npig[a, out["gt_labels"][b, gi]] += 1
    return oracle.accumulate_ap(recs, npig, thrs, max_dets, nc), npig


@pytest.mark.parametrize("quantise", [False, True])
def test_device_sweep_records_and_accumulate_kernel(quantise):
    """a9 on the device: the records the library appends per batch (zero torch ops) decode to the oracle's per-detection
    match bits, and btpost_sweep_accumulate (radix sort + scans + 101-point lookup) reproduces the oracle's numpy
    restatement of COCOeval.accumulate BIT FOR BIT (doubles), also when scores tie across images (quantised scores: the
    global order then hangs on the (image, rank) tie-break) and when batches arrive out of order."""
    kw = dict(max_det=100, gt_mode=1)
    B, S, nb = 4, 160, 5
    sweep = DeviceSweep(3, oracle.iou_thresholds(), (1, 10, 100), capacity=4096, max_det_per_image=100, device="cuda:0")
    cfg = PostConfig(batch=B, img_size=S, max_det=100, gt_mode=1, with_coco=True)
    pp = PostProcessor(cfg, "cuda:0", sweep=sweep)
    outs, offs = [], []
    for i in (3, 0, 4, 1, 2):                             # batches in scrambled order: the result must not depend on it
        batch = helpers.make(batch=B, img_size=S, seed=31, image_offset=B * i)
        if quantise:
            batch["head"][:, 4:7] = np.round(batch["head"][:, 4:7] * 16) / 16
        if i == 1:
            batch["head"][2, 4:7] = 0.0                   # an image without candidates
        ref = oracle.run_pipeline(batch, img_size=S, **kw)
        d = helpers.to_dev(batch, "cuda:0")
        out = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"], image_offset=B * i)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(out["dt_match"].cpu().numpy(), ref["dt_match"])
        outs.append(ref); offs.append(B * i)
    # ---- records
    n = int(sweep.hdr[0])
    assert n == sum(int(o["det_count"].sum()) for o in outs)
    rec = decode_records(sweep.records[:n], 10)
    for ref, off in zip(outs, offs):
        for b in range(B):
            k = int(ref["det_count"][b])
            sel = np.nonzero(rec["image"] == off + b)[0]
            assert len(sel) == k
            sel = sel[np.argsort(rec["rank"][sel])]
            np.testing.assert_array_equal(rec["rank"][sel], np.arange(k))
            assert rec["score"][sel].tobytes() == ref["dets"][b, :k, 4].tobytes()
            lab = ref["dets"][b, :k, 5].astype(np.int64)
            np.testing.assert_array_equal(rec["label"][sel], lab)
            np.testing.assert_array_equal(rec["class_rank"][sel], [int((lab[:j] == lab[j]).sum()) for j in range(k)])
            np.testing.assert_array_equal(rec["matched"][sel], np.moveaxis(ref["dt_match"][b][:, :, :k] > 0, 2, 0))
            np.testing.assert_array_equal(rec["ignored"][sel], np.moveaxis(ref["dt_ignore"][b][:, :, :k] > 0, 2, 0))
    # ---- header + accumulate
    want, npig = _oracle_ap(outs, offs)
    res = sweep.finish()
    assert res["n_images"] == nb * B and res["n_records"] == n
    np.testing.assert_array_equal(res["npig"], npig)
    np.testing.assert_array_equal(res["precision"], want["precision"])      # float64, bit for bit
    np.testing.assert_array_equal(res["recall"], want["recall"])
    for k in ("map", "map_50", "map_75", "mar_1", "mar_10", "mar_100", "map_small", "map_medium", "map_large"):
        assert res[k] == want[k], k
    assert want["map_50"] > 0.05
    np.testing.assert_array_equal(res["cm"].numpy(), sum(o["cm"] for o in outs))
    assert res["seg_dice"] == pytest.approx(float(np.mean([o["seg_dice"] for o in outs])), rel=1e-6)
    assert res["uni_iou"] == pytest.approx(float(np.mean([o["uni_iou"] for o in outs])), rel=1e-6)
    # second finish() on the untouched ring gives the same tables (the sort works on a copy)
    np.testing.assert_array_equal(sweep.finish()["precision"], want["precision"])


def test_device_sweep_through_pipeline_drop_flag_and_overflow():
    """Sweep records from captured steps replayed with several batches in flight (image index through the device-side
    `image_base`), the v2 `drop_gt_no_cand` rule in the GT counts, and the ring-overflow report."""
    B, S, depth = 4, 160, 3
    for drop, auto in ((False, False), (True, False), (False, True)):   # auto: the images are numbered on the device
        sweep = DeviceSweep(3, oracle.iou_thresholds(), (1, 10, 100), capacity=8192, max_det_per_image=100, device="cuda:0")
        cfg = PostConfig(batch=B, img_size=S, max_det=100, gt_mode=1, with_coco=True, drop_gt_no_cand=drop)
        batches = [helpers.make(batch=B, img_size=S, seed=91, image_offset=B * i) for i in range(6)]
        batches[2]["head"][1, 4:7] = 0.0
        w, bias = helpers.to_dev(batches[0], "cuda:0")["proj_weight"], float(batches[0]["proj_bias"])
        pipe = Pipeline(cfg, "cuda:0", depth=depth, proj_weight=w, proj_bias=bias, sweep=sweep, auto_image_offset=auto)
        outs, offs = [], []
        for i, bt in enumerate(batches):
            d = helpers.to_dev(bt, "cuda:0")
            pipe.submit(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], image_offset=None if auto else B * i)
            outs.append(oracle.run_pipeline(bt, img_size=S, max_det=100, gt_mode=1)); offs.append(B * i)
        pipe.join()
        torch.cuda.synchronize()
        want, npig = _oracle_ap(outs, offs, drop=drop)
        res = sweep.finish()
        np.testing.assert_array_equal(res["npig"], npig)
        np.testing.assert_array_equal(res["precision"], want["precision"])
        assert res["n_images"] == 6 * B
    small = DeviceSweep(3, oracle.iou_thresholds(), (1, 10, 100), capacity=16, max_det_per_image=100, device="cuda:0")
    pp = PostProcessor(cfg, "cuda:0", sweep=small)
    d = helpers.to_dev(batches[0], "cuda:0")
    pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"])
    with pytest.raises(RuntimeError, match="ring too small"):
        small.finish()


@pytest.mark.parametrize("case", [dict(n_img=40, K=12, nc=3, T=10, max_dets=(1, 10, 100), q=8),
                                  dict(n_img=700, K=40, nc=5, T=10, max_dets=(1, 5, 20), q=4),       # image index needs two radix passes
                                  dict(n_img=9, K=300, nc=2, T=3, max_dets=(3, 100, 300), q=64),     # rank needs two radix passes
                                  dict(n_img=64, K=30, nc=1, T=16, max_dets=(100,), q=2)])           # one class, 16 thresholds, masses of ties
def test_accumulate_kernel_fuzz_against_oracle(case):
    """btpost_sweep_accumulate on RANDOM records (random match / ignore bits, heavily tied scores, classes without GT or
    without detections, more images than one radix digit, more detections per image than one radix digit) against the
    oracle's numpy restatement of COCOeval.accumulate: the float64 tables must be identical."""
    from test_sweep import encode_records
    from btpost import _lib
    n_img, K, nc, T, max_dets, q = (case[k] for k in ("n_img", "K", "nc", "T", "max_dets", "q"))
    rng = np.random.default_rng(n_img * 1000 + K)
    thrs = np.linspace(0.5, 0.95, T) if T > 1 else np.array([0.5])
    dets = np.zeros((n_img, K, 6), np.float32)
    cnt = rng.integers(0, K + 1, n_img).astype(np.int32)
    dt_match = np.zeros((n_img, 4, T, K), np.int32)
    dt_ignore = np.zeros((n_img, 4, T, K), np.uint8)
    recs = []
    for b in range(n_img):
        k = int(cnt[b])
        sc = np.sort((rng.integers(1, q + 1, k) / q).astype(np.float32))[::-1]
        dets[b, :k, 4] = sc
        dets[b, :k, 5] = rng.integers(0, nc, k)
        dt_match[b, :, :, :k] = rng.integers(0, 2, (4, T, k)) * rng.integers(1, 4, (4, T, k))
        dt_ignore[b, :, :, :k] = rng.integers(0, 4, (4, T, k)) == 0
        recs.append(dict(labels=dets[b, :k, 5].astype(np.int64), scores=dets[b, :k, 4], matched=dt_match[b][:, :, :k] > 0,
                         ignored=dt_ignore[b][:, :, :k] > 0))
    npig = rng.integers(0, 50, (4, nc)).astype(np.int64)
    npig[:, rng.integers(0, nc)] *= rng.integers(0, 2)                      # sometimes a class without any GT
    want = oracle.accumulate_ap(recs, npig, thrs, max_dets, nc)
    out = dict(det_count=cnt, dets=dets, dt_match=dt_match, dt_ignore=dt_ignore)
    raw = encode_records(out, 0, T)
    perm = rng.permutation(len(raw))                                        # the ring order is whatever the atomics made it
    raw = raw[perm]
    sweep = DeviceSweep(nc, thrs, max_dets, capacity=len(raw) + 5, max_det_per_image=K, device="cuda:0")
    sweep.records[:len(raw)].copy_(torch.from_numpy(raw.view(np.uint8).reshape(-1, 32)))
    hdr = np.zeros(sweep.hdr.numel(), np.int64)
    hdr[_lib.SWEEP_N_RECORDS], hdr[_lib.SWEEP_N_IMAGES], hdr[_lib.SWEEP_CAPACITY] = len(raw), n_img, len(raw) + 5
    hdr[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64].reshape(4, 16)[:, :nc] = npig
    sweep.hdr.copy_(torch.from_numpy(hdr))
    res = sweep.finish()
    np.testing.assert_array_equal(res["precision"], want["precision"])
    np.testing.assert_array_equal(res["recall"], want["recall"])
    for k in ("map", "map_50", "map_75", "map_small", "map_medium", "map_large"):
        assert res[k] == want[k], k
