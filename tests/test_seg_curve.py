"""CPU: binned PR / ROC curves of the projector probabilities (btpost_seg_curve, btpost.segcurve) -- the numpy
restatement of tests/seg_curve_oracle.py against a literal restatement of torchmetrics' binned update, the curve formulas
against an independent Mann-Whitney AUROC and a sort-based AP, the arguments btpost_seg_curve rejects before any CUDA
call, and the curve state riding in the existing header all-reduce of a 2-rank gloo merge."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import seg_curve_oracle as sco
from btpost import _lib, segcurve
from btpost.api import PostConfig
from btpost.sweep import HDR, REC_BYTES, merge_sweeps
from test_sweep import _free_port


def torchmetrics_confmat(p, gt, thr):
    """torchmetrics' _binary_precision_recall_curve_update_vectorized, written out: [T, 2, 2] indexed [k, target, pred]."""
    p, thr = torch.from_numpy(np.asarray(p, np.float32).reshape(-1)), torch.from_numpy(np.asarray(thr, np.float32))
    t = torch.from_numpy((np.asarray(gt) != 0).reshape(-1)).long()
    T = len(thr)
    preds_t = (p.unsqueeze(-1) >= thr.unsqueeze(0)).long()
    unique_mapping = preds_t + 2 * t.unsqueeze(-1) + 4 * torch.arange(T)
    bins = torch.bincount(unique_mapping.flatten(), minlength=4 * T)
    return bins.reshape(T, 2, 2).numpy()


def fuzz_case(rng, T):
    """Probabilities that sit on the thresholds, on their fp32 neighbours, at 0, 1 and NaN, plus uniform ones; duplicate
    thresholds; GT that is mixed, all background or all foreground."""
    thr = np.sort(rng.random(T).astype(np.float32))
    thr[rng.integers(T, size=T // 4)] = thr[rng.integers(T)]                  # duplicates
    thr[0], thr[-1] = (np.float32(0.0), np.float32(1.0)) if rng.random() < 0.5 else (thr[0], thr[-1])
    thr = np.sort(thr)
    on = thr[rng.integers(T, size=400)]
    p = np.concatenate([on, np.nextafter(on, np.float32(2)), np.nextafter(on, np.float32(-1)), rng.random(600).astype(np.float32),
                        np.float32([0.0, 1.0, np.nan, 0.0, 1.0, np.nan])])
    p = np.clip(p, 0, 1).astype(np.float32)
    p[-6:] = np.float32([0.0, 1.0, np.nan, 0.0, 1.0, np.nan])
    kind = rng.integers(3)
    gt = rng.random(p.size) < 0.3 if kind == 0 else np.zeros(p.size, bool) if kind == 1 else np.ones(p.size, bool)
    return rng.permutation(p), gt, thr


@pytest.mark.parametrize("T", [2, 3, 101, 1024])
def test_restatement_equals_torchmetrics_binned_update(T):
    rng = np.random.default_rng(T)
    for _ in range(8):
        p, gt, thr = fuzz_case(rng, T)
        h = sco.hist_from_probs(p, gt, thr)
        assert h.sum() == p.size and h[1].sum() == gt.sum()
        np.testing.assert_array_equal(segcurve.confmat(h), torchmetrics_confmat(p, gt, thr))
    lin = segcurve.thresholds(T)                                           # torchmetrics' own thresholds=T
    p, gt, _ = fuzz_case(rng, T)
    np.testing.assert_array_equal(segcurve.confmat(sco.hist_from_probs(p, gt, lin)), torchmetrics_confmat(p, gt, lin))


def test_restatement_from_logits_uses_the_soft_dice_probability():
    rng = np.random.default_rng(3)
    x = np.concatenate([rng.normal(0, 6, 5000), [-87.5, -87.0, 0.0, 88.0, -1e-9, 1e-9]]).astype(np.float32).reshape(1, 1, -1)
    gt = rng.random(x.shape) < 0.5
    thr = segcurve.thresholds(101)
    np.testing.assert_array_equal(sco.seg_curve_hist(x, gt, thr),
                                  sco.hist_from_probs(sco.soft_prob(x), gt, thr))
    assert sco.soft_prob(np.float32([-87.5]))[0] == 0.0


def mann_whitney(p, t):
    pos, neg = p[t].astype(np.float64), p[~t].astype(np.float64)
    gt_ = (pos[:, None] > neg[None, :]).sum()
    eq = (pos[:, None] == neg[None, :]).sum()
    return (gt_ + 0.5 * eq) / (len(pos) * len(neg))


def sorted_ap(p, t):
    """Step-wise AP: walk the distinct scores from high to low, precision at each times the recall it adds."""
    ap, tp, fp, npos = 0.0, 0, 0, int(t.sum())
    for v in np.unique(p)[::-1]:
        sel = p == v
        dtp = int((t & sel).sum())
        tp, fp = tp + dtp, fp + int((~t & sel).sum())
        ap += dtp / npos * tp / (tp + fp)
    return ap


@pytest.mark.parametrize("seed", range(6))
def test_formulas_equal_mann_whitney_auroc_and_sorted_ap(seed):
    """With the thresholds at every distinct p plus one above the largest, the binned curves are the exact ones."""
    rng = np.random.default_rng(100 + seed)
    n, levels = int(rng.integers(50, 3000)), int(rng.integers(5, 1000))
    p = (rng.integers(0, levels, n) / np.float32(levels + 1)).astype(np.float32)   # ties, all below 1
    t = rng.random(n) < rng.uniform(0.05, 0.9) * np.where(p > 0.5, 1.0, 0.5)
    t[:2] = [True, False]
    thr = np.concatenate([np.unique(p), [np.nextafter(p.max(), np.float32(2))]]).astype(np.float32)
    m = segcurve.curve_metrics(segcurve.confmat(sco.hist_from_probs(p, t, thr)), thr)
    assert m["auroc"] == pytest.approx(mann_whitney(p, t), abs=1e-12, rel=0)
    assert m["ap"] == pytest.approx(sorted_ap(p, t), abs=1e-12, rel=0)
    precision, recall, th = m["pr_curve"]
    assert precision[-1] == 1.0 and recall[-1] == 0.0 and len(precision) == len(thr) + 1 and (th == thr).all()
    fpr, tpr, rth = m["roc"]
    assert (rth == thr[::-1]).all() and fpr[0] == 0.0 and tpr[-1] == 1.0 and fpr[-1] == 1.0


def test_zero_division_conventions():
    # every pixel background: recall and tpr 0 / 0 -> 0; precision 0 / 0 (nothing predicted) -> 1
    thr = np.float32([0.0, 0.5, 1.0])
    m = segcurve.curve_metrics(segcurve.confmat(sco.hist_from_probs(np.float32([0.2, 0.3]), [0, 0], thr)), thr)
    precision, recall, _ = m["pr_curve"]
    np.testing.assert_array_equal(precision, [0.0, 1.0, 1.0, 1.0])
    np.testing.assert_array_equal(recall, [0.0, 0.0, 0.0, 0.0])
    np.testing.assert_array_equal(m["roc"][1], [0.0, 0.0, 0.0])
    np.testing.assert_array_equal(m["roc"][0], [0.0, 0.0, 1.0])
    assert m["ap"] == 0.0 and m["auroc"] == 0.0


def test_threshold_specs():
    np.testing.assert_array_equal(segcurve.thresholds(101), torch.linspace(0, 1, 101).numpy())
    assert segcurve.thresholds([0, 0.5, 0.5, 1]).dtype == np.float32
    for bad in (1, 1025, 0, [0.5], [0.2, 0.1], [0.0, 1.5], [-0.1, 0.5], [0.0, float("nan")], list(np.linspace(0, 1, 1025))):
        with pytest.raises(ValueError):
            segcurve.thresholds(bad)
    assert PostConfig(batch=1).seg_curve is None


def _params(S=160, B=2):
    p = _lib.BtParams()
    p.batch, p.nc, p.nm, p.reg_max, p.max_det, p.max_gt = B, 3, 32, 16, 300, 32
    p.num_anchors = sum((S // s) ** 2 for s in (8, 16, 32))
    p.img_h = p.img_w = S
    p.proto_h = p.proto_w = S // 4
    p.num_iou_thrs = 10
    return p


def test_seg_curve_argument_validation_without_gpu():
    """Every error of btpost_seg_curve is returned before any CUDA call (fake device pointers, host thresholds)."""
    L = _lib.load()
    p = _params()
    n = C.c_size_t()
    assert L.btpost_workspace_bytes(C.byref(p), C.byref(n)) == 0
    ws = n.value

    def call(thr=(0.0, 0.5, 1.0), T=None, hist=4096, params=p, ws_ptr=1 << 20, nbytes=ws):
        arr = None if thr is None else (C.c_float * max(len(thr), 1))(*thr)
        return L.btpost_seg_curve(None if params is None else C.byref(params), ws_ptr, nbytes, arr,
                                  len(thr) if T is None else T, hist, None)
    assert call(thr=None, T=3) == -1 and call(hist=None) == -1
    assert call(thr=(0.5,)) == -1 and call(thr=tuple(np.linspace(0, 1, 1025, dtype=np.float32).tolist())) == -1
    assert call(T=0) == -1 and call(T=-2) == -1
    assert call(thr=(0.0, -1e-8, 1.0)) == -1 and call(thr=(0.0, 1.0000001)) == -1
    assert call(thr=(0.0, float("nan"), 1.0)) == -1 and call(thr=(0.0, 0.6, 0.5)) == -1
    assert call(hist=4100) == -4
    assert call(params=None) == -1
    bad = _params()
    bad.batch = 0
    assert call(params=bad) == -1
    bad = _params()
    bad.img_h = bad.img_w = 650
    assert call(params=bad) == -2
    assert call(ws_ptr=None) == -1 and call(ws_ptr=(1 << 20) + 16) == -4 and call(nbytes=ws - 1) == -3
    assert _lib.BT_MAX_CURVE_THRS == 1024 == segcurve.MAX_THRESHOLDS


# ---------------------------------------------------------------------------------------------- 2-rank merge (gloo)
RECORDS = ((7, 2), (3, 9))                   # [rank][state]: ragged record counts
T_CURVE = 101


def _shard(rank):
    rng = np.random.default_rng(40 + rank)
    hdrs, rings = [], []
    for n in RECORDS[rank]:
        h = rng.integers(0, 1 << 40, HDR).astype(np.int64)
        h[_lib.SWEEP_N_RECORDS] = n
        ring = np.zeros((n + 3 * rank, REC_BYTES), np.uint8)
        ring[:n] = rng.integers(0, 256, (n, REC_BYTES))
        hdrs.append(h)
        rings.append(ring)
    curve = rng.integers(0, 1 << 40, (2, T_CURVE + 1)).astype(np.int64)
    return hdrs, rings, curve


def _merge_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        calls = {"all_reduce": 0, "all_gather_into_tensor": 0, "other": 0}

        def counted(name, fn):
            def wrap(*a, **k):
                calls[name] += 1
                return fn(*a, **k)
            return wrap
        dist.all_reduce = counted("all_reduce", dist.all_reduce)
        dist.all_gather_into_tensor = counted("all_gather_into_tensor", dist.all_gather_into_tensor)
        for name in ("all_gather", "broadcast", "reduce", "gather", "scatter", "reduce_scatter"):
            setattr(dist, name, counted("other", getattr(dist, name)))
        hdrs, rings, curve = _shard(rank)
        got = []
        for states in (1, 2):                 # one state (the detection sweep alone) and two
            h = [torch.from_numpy(x.copy()) for x in hdrs[:states]]
            c = torch.from_numpy(curve.copy())
            before = dict(calls)
            ns, merged = merge_sweeps(h, [torch.from_numpy(r) for r in rings[:states]], extra=(c,))
            got.append((ns, [m.numpy().copy() for m in merged], [x.numpy().copy() for x in h], c.numpy().copy(),
                        {k: calls[k] - before[k] for k in calls}))
        if rank == 1:
            q.put(got)
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_merge_carries_the_curve_in_the_header_all_reduce():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_merge_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    shards = [_shard(r) for r in range(world)]
    for states, (ns, merged, hdrs, curve, calls) in zip((1, 2), got):
        assert calls == {"all_reduce": 1, "all_gather_into_tensor": 2, "other": 0}   # the collectives of a merge without it
        np.testing.assert_array_equal(curve, shards[0][2] + shards[1][2])
        for s in range(states):
            assert ns[s] == [RECORDS[r][s] for r in range(world)]
            np.testing.assert_array_equal(hdrs[s], shards[0][0][s] + shards[1][0][s])
            np.testing.assert_array_equal(merged[s], np.concatenate([shards[r][1][s][:RECORDS[r][s]] for r in range(world)]))
