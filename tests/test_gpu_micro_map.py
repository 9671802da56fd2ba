"""-m gpu: the class-agnostic state (BtIOMicro.micro_sweep) written by match_kernel and the score table of
btpost_sweep_accumulate_ext, against the CPU restatements of tests/micro_oracle.py."""
import numpy as np
import pytest
import torch

import helpers
import micro_oracle
from btpost import Pipeline, PostConfig, PostProcessor, _lib
from btpost.sweep import DeviceSweep, decode_records
from oracle import oracle

pytestmark = pytest.mark.gpu

MAX_DETS = (1, 10, 100)
CLASS_AWARE_OUTS = ("dets", "det_count", "dt_match", "dt_ignore", "gt_ignore")


@pytest.mark.parametrize("S,B", [(160, 4), (640, 2), (1024, 1)])
def test_micro_records_and_tables_against_oracle(S, B):
    """The micro records decode to the oracle's class-agnostic matching (match / ignore bits, rank, score), the micro
    tables equal accumulate_ap(nc=1) BIT FOR BIT, every score table equals the numpy restatement bit for bit, and the
    class-aware outputs, records and tables are the same as without the micro state."""
    thrs = oracle.iou_thresholds()
    kw = dict(max_det=100, gt_mode=1)
    cfg = PostConfig(batch=B, img_size=S, max_det=100, gt_mode=1, with_coco=True)
    sweeps = [DeviceSweep(3, thrs, MAX_DETS, capacity=8192, max_det_per_image=100, device="cuda:0", micro=m) for m in (False, True)]
    procs = [PostProcessor(cfg, "cuda:0", sweep=s) for s in sweeps]
    outs, got = [], [[], []]
    for i in range(2):
        batch = helpers.make(batch=B, img_size=S, seed=41 + S, image_offset=B * i)
        if i == 1:
            batch["head"][0, 4:7] = batch["head"][0, [5, 6, 4]]      # class scores rotated: wrong-class boxes on the GTs
        outs.append(oracle.run_pipeline(batch, img_size=S, with_instances=False, with_masks_out=False, **kw))
        d = helpers.to_dev(batch, "cuda:0")
        for j, pp in enumerate(procs):
            o = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"], image_offset=B * i)
            torch.cuda.synchronize()
            got[j].append({k: o[k].cpu().numpy() for k in CLASS_AWARE_OUTS})
        np.testing.assert_array_equal(got[1][-1]["dt_match"], outs[-1]["dt_match"])
    for a, b in zip(*got):
        for k in CLASS_AWARE_OUTS:
            assert a[k].tobytes() == b[k].tobytes(), k
    n = int(sweeps[0].hdr[0])
    assert int(sweeps[1].hdr[0]) == n and sweeps[0].records[:n].cpu().numpy().tobytes() == sweeps[1].records[:n].cpu().numpy().tobytes()
    # ---- micro records
    mh = sweeps[1].micro_hdr.cpu().numpy()
    assert mh[_lib.SWEEP_N_RECORDS] == n and mh[_lib.SWEEP_N_IMAGES] == 2 * B
    rec = decode_records(sweeps[1].micro_records[:n], 10)
    for i, out in enumerate(outs):
        for b in range(B):
            want, dm, di, _ = micro_oracle.micro_records(out, b, thrs)
            k = len(want["labels"])
            sel = np.nonzero(rec["image"] == B * i + b)[0]
            sel = sel[np.argsort(rec["rank"][sel])]
            np.testing.assert_array_equal(rec["rank"][sel], np.arange(k))
            np.testing.assert_array_equal(rec["class_rank"][sel], np.arange(k))
            assert not rec["label"][sel].any()
            assert rec["score"][sel].tobytes() == out["dets"][b, :k, 4].tobytes()
            np.testing.assert_array_equal(rec["matched"][sel], np.moveaxis(dm > 0, 2, 0))
            np.testing.assert_array_equal(rec["ignored"][sel], np.moveaxis(di > 0, 2, 0))
    # ---- tables
    want, npig, mrecs = micro_oracle.micro_ap(outs, thrs, MAX_DETS)
    r0, r1 = sweeps[0].finish(extended_summary=True), sweeps[1].finish(extended_summary=True)
    np.testing.assert_array_equal(mh[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64: 16], npig[:, 0])
    assert r1["micro_precision"].tobytes() == want["precision"].tobytes()
    assert r1["micro_recall"].tobytes() == want["recall"].tobytes()
    for k in ("map", "map_50", "map_75", "map_small", "map_medium", "map_large", "mar_1", "mar_10", "mar_100"):
        assert r1[f"micro_{k}"] == want[k], k
    assert "micro_map_per_class" not in r1
    assert r1["micro_scores"].tobytes() == micro_oracle.score_table(mrecs, npig, thrs, MAX_DETS, 1).tobytes()
    for k in ("precision", "recall", "scores", "map", "map_50", "map_per_class"):
        assert np.asarray(r0[k]).tobytes() == np.asarray(r1[k]).tobytes(), k
    drec = micro_oracle.records_from_ring(decode_records(sweeps[0].records[:n], 10))
    assert r0["scores"].tobytes() == micro_oracle.score_table(drec, r0["npig"], thrs, MAX_DETS, 3).tobytes()
    assert "scores" not in sweeps[1].finish() and r1["micro_map_50"] > 0


def test_seg_map_score_table():
    """The score table of the segmentation-mAP state (one record per image) equals the numpy restatement bit for bit."""
    thrs = oracle.iou_thresholds()
    B, S = 8, 160
    sweep = DeviceSweep(3, thrs, MAX_DETS, capacity=4096, max_det_per_image=100, device="cuda:0", seg_map_capacity=64)
    cfg = PostConfig(batch=B, img_size=S, max_det=100, gt_mode=1, with_coco=True, with_seg_map=True)
    pp = PostProcessor(cfg, "cuda:0", sweep=sweep)
    for i in range(3):
        d = helpers.to_dev(helpers.make(batch=B, img_size=S, seed=5 + i, image_offset=B * i), "cuda:0")
        pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"], image_offset=B * i)
    torch.cuda.synchronize()
    n = int(sweep.seg_hdr[0])
    recs = micro_oracle.records_from_ring(decode_records(sweep.seg_records[:n], 10))
    npig = sweep.seg_hdr[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64: 16].cpu().numpy()[:, None]
    res = sweep.finish(extended_summary=True)
    want = micro_oracle.score_table(recs, npig, thrs, MAX_DETS, 1)
    assert res["seg_map_scores"].tobytes() == want.tobytes()
    assert (want[:, 0, 0, 0, 0] > 0).all()


@pytest.mark.parametrize("case", [dict(n_img=40, K=12, nc=3, T=10, max_dets=(1, 10, 100), q=8),
                                  dict(n_img=700, K=40, nc=5, T=10, max_dets=(1, 5, 20), q=4),
                                  dict(n_img=9, K=300, nc=2, T=3, max_dets=(3, 100, 300), q=64),
                                  dict(n_img=64, K=30, nc=1, T=16, max_dets=(100,), q=2),
                                  dict(n_img=2000, K=3, nc=2, T=1, max_dets=(1, 2), q=3),    # many chunks per class
                                  dict(n_img=300, K=20, nc=3, T=10, max_dets=(1, 10, 100), q=1 << 22)])   # continuous scores
def test_score_table_fuzz(case):
    """btpost_sweep_accumulate_ext on random records (the accumulate fuzz cases, plus ignored records at the head of
    sequences and a class without GT): the score table equals the numpy restatement bit for bit, and precision / recall
    equal those of btpost_sweep_accumulate."""
    from test_sweep import encode_records
    n_img, K, nc, T, max_dets, q = (case[k] for k in ("n_img", "K", "nc", "T", "max_dets", "q"))
    rng = np.random.default_rng(n_img * 1000 + K + 1)
    thrs = np.linspace(0.5, 0.95, T) if T > 1 else np.array([0.5])
    dets = np.zeros((n_img, K, 6), np.float32)
    cnt = rng.integers(0, K + 1, n_img).astype(np.int32)
    cnt[:3] = np.maximum(cnt[:3], 1)
    dt_match = np.zeros((n_img, 4, T, K), np.int32)
    dt_ignore = np.zeros((n_img, 4, T, K), np.uint8)
    recs = []
    for b in range(n_img):
        k = int(cnt[b])
        dets[b, :k, 4] = np.sort((rng.integers(1, q + 1, k) / q).astype(np.float32))[::-1]
        dets[b, :k, 5] = rng.integers(0, nc, k)
        dt_match[b, :, :, :k] = rng.integers(0, 2, (4, T, k)) * rng.integers(1, 4, (4, T, k))
        dt_ignore[b, :, :, :k] = rng.integers(0, 4, (4, T, k)) == 0
        if b < 3:   # the head of class b % nc's sequence (score above every other), ignored at every (area, threshold)
            dets[b, 0, 4], dets[b, 0, 5] = 2.0 - 0.25 * b, b % nc
            dt_ignore[b, :, :, :1] = 1
        recs.append(dict(labels=dets[b, :k, 5].astype(np.int64), scores=dets[b, :k, 4], matched=dt_match[b][:, :, :k] > 0,
                         ignored=dt_ignore[b][:, :, :k] > 0))
    npig = rng.integers(1, 50, (4, nc)).astype(np.int64)
    if nc > 1:
        npig[:, -1] = 0
    raw = encode_records(dict(det_count=cnt, dets=dets, dt_match=dt_match, dt_ignore=dt_ignore), 0, T)
    raw = raw[rng.permutation(len(raw))]
    sweep = DeviceSweep(nc, thrs, max_dets, capacity=len(raw) + 5, max_det_per_image=K, device="cuda:0")
    sweep.records[:len(raw)].copy_(torch.from_numpy(raw.view(np.uint8).reshape(-1, 32)))
    hdr = np.zeros(sweep.hdr.numel(), np.int64)
    hdr[_lib.SWEEP_N_RECORDS], hdr[_lib.SWEEP_N_IMAGES], hdr[_lib.SWEEP_CAPACITY] = len(raw), n_img, len(raw) + 5
    hdr[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64].reshape(4, 16)[:, :nc] = npig
    sweep.hdr.copy_(torch.from_numpy(hdr))
    res = sweep.finish(extended_summary=True)
    want = micro_oracle.score_table(recs, npig, thrs, max_dets, nc)
    assert res["scores"].tobytes() == want.tobytes()
    for b in range(min(3, n_img)):   # recall 0 is reached at the sequence's first record, ignored or not
        c = b % nc
        if b < nc:
            sel = npig[:, c] > 0
            assert (res["scores"][:, 0, c][:, sel] == 2.0 - 0.25 * b).all()
    ap = oracle.accumulate_ap(recs, npig, thrs, max_dets, nc)
    assert res["precision"].tobytes() == ap["precision"].tobytes() and res["recall"].tobytes() == ap["recall"].tobytes()


def test_pipeline_with_micro_state_and_overflow():
    """Captured steps replayed with several batches in flight and images numbered on the device: the class-aware keys and
    records are the same with and without micro=True, the micro tables equal the oracle's; a micro ring that is too
    small raises like the others."""
    B, S, depth = 4, 160, 3
    thrs = oracle.iou_thresholds()
    cfg = PostConfig(batch=B, img_size=S, max_det=100, gt_mode=1, with_coco=True)
    batches = [helpers.make(batch=B, img_size=S, seed=91, image_offset=B * i) for i in range(5)]
    w, bias = helpers.to_dev(batches[0], "cuda:0")["proj_weight"], float(batches[0]["proj_bias"])
    results, rings = [], []
    for micro in (False, True):
        sweep = DeviceSweep(3, thrs, MAX_DETS, capacity=8192, max_det_per_image=100, device="cuda:0", micro=micro)
        pipe = Pipeline(cfg, "cuda:0", depth=depth, proj_weight=w, proj_bias=bias, sweep=sweep, auto_image_offset=True)
        for bt in batches:
            d = helpers.to_dev(bt, "cuda:0")
            pipe.submit(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"])
        pipe.join()
        torch.cuda.synchronize()
        n = int(sweep.hdr[0])
        rings.append(sorted(bytes(r) for r in sweep.records[:n].cpu().numpy()))
        results.append(sweep.finish())
    assert rings[0] == rings[1]
    for k, v in results[0].items():
        if isinstance(v, torch.Tensor):
            v = v.numpy()
        got = results[1][k].numpy() if isinstance(results[1][k], torch.Tensor) else results[1][k]
        assert np.asarray(v).tobytes() == np.asarray(got).tobytes(), k
    outs = [oracle.run_pipeline(bt, img_size=S, max_det=100, gt_mode=1, with_instances=False, with_masks_out=False) for bt in batches]
    want, _, _ = micro_oracle.micro_ap(outs, thrs, MAX_DETS)
    assert results[1]["micro_precision"].tobytes() == want["precision"].tobytes()
    assert results[1]["n_micro_records"] == results[1]["n_records"]
    small = DeviceSweep(3, thrs, MAX_DETS, capacity=16, max_det_per_image=100, device="cuda:0", micro=True)
    pp = PostProcessor(cfg, "cuda:0", sweep=small)
    d = helpers.to_dev(batches[0], "cuda:0")
    pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"])
    torch.cuda.synchronize()
    assert int(small.micro_hdr[_lib.SWEEP_N_RECORDS]) > 16
    with pytest.raises(RuntimeError, match="DeviceSweep ring too small"):
        small.finish()
    small.hdr[_lib.SWEEP_N_RECORDS] = 0                               # the detection ring alone within its capacity
    with pytest.raises(RuntimeError, match="class-agnostic ring too small"):
        small.finish()
