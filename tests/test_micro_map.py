"""CPU: the class-agnostic box mAP (BtIOMicro.micro_sweep, torchmetrics average="micro") and COCOeval.accumulate's score
table -- the ABI layout of the new struct, its argument validation (before any CUDA call), the oracle restatements, and
the merge of three sweep states across a 2-rank gloo group with the collectives of one."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import micro_oracle
from btpost import _lib, synth
from btpost.sweep import HDR, decode_records, merge_sweeps
from oracle import oracle
from test_seg_map_sweep import _det_shard, _params, _seg_shard
from test_sweep import _free_port, encode_records

ROOT = Path(__file__).resolve().parents[1]
KW = dict(conf_thres=0.05, iou_thres=0.6, max_det=100, gt_mode=1, with_instances=False, with_masks_out=False)


def test_btio_micro_layout(tmp_path):
    """BtParams keeps its size (io_micro takes the reserved word); BtIOMicro = BtIOSoftDice + one pointer."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "btpost.h"\nint main(){'
                   'printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(BtParams), offsetof(BtParams, io_soft_dice),'
                   'offsetof(BtParams, io_micro), sizeof(BtIO), sizeof(BtIOSoftDice), sizeof(BtIOMicro),'
                   'offsetof(BtIOMicro, micro_sweep));return 0;}')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(_lib.BtParams), _lib.BtParams.io_soft_dice.offset, _lib.BtParams.io_micro.offset,
                   C.sizeof(_lib.BtIO), C.sizeof(_lib.BtIOSoftDice), C.sizeof(_lib.BtIOMicro), _lib.BtIOMicro.micro_sweep.offset]
    assert got[0] == 272 and got[2] == got[1] + 4 and got[2] + 4 == got[0]   # the size BtParams had with reserved[1]
    assert got[4] == 376                                                       # BtIOSoftDice unchanged
    assert got[5] == got[4] + 8 and got[6] == got[4]


def test_micro_sweep_argument_validation_without_gpu():
    """io_micro must be 0 or 1; the state needs the COCO matching (dt_match) and 16-byte alignment.  Checked by the NMS /
    matching stage and by btpost_run before any CUDA call."""
    L = _lib.load()
    p, ws = _params()
    io = _lib.BtIOMicro()
    for f in ("head", "protos", "masks_gt", "proj_weight", "dets", "det_count", "det_coeff", "det_keep", "det_anchor", "n_cand",
              "gt_count", "gt_boxes", "gt_boxes_raw", "gt_labels", "cm", "cm_pos"):
        setattr(io, f, 4096)
    nms = lambda: L.btpost_nms_match(C.byref(p), C.cast(C.byref(io), C.POINTER(_lib.BtIO)), C.c_void_p(256), ws, None)
    run = lambda: L.btpost_run(C.byref(p), C.cast(C.byref(io), C.POINTER(_lib.BtIO)), C.c_void_p(256), ws, None)
    p.io_micro = 2
    assert nms() == -1 and run() == -1
    p.io_micro = 1
    io.micro_sweep = 8192                                            # no dt_match
    assert nms() == -1 and run() == -1
    io.dt_match, io.micro_sweep = 4096, 8192 + 8                     # misaligned state
    assert nms() == -4 and run() == -4


# ---------------------------------------------------------------------------------------------- oracle restatements
def _oracle(n_images, nc=3, seed=77):
    cfg = synth.SynthConfig(batch=n_images, img_size=160, seed=seed, nc=nc)
    return oracle.run_pipeline(synth.make_batch(cfg), img_size=160, nc=nc, **KW)


def _class_aware(out, nc):
    recs, npig = [], np.zeros((4, nc), np.int64)
    for b in range(len(out["det_count"])):
        k, g = int(out["det_count"][b]), int(out["gt_count"][b])
        recs.append(dict(labels=out["dets"][b, :k, 5].astype(np.int64), scores=out["dets"][b, :k, 4],
                         matched=out["dt_match"][b][:, :, :k] > 0, ignored=out["dt_ignore"][b][:, :, :k] > 0))
        for a in range(4):
            for gi in range(g):
                npig[a, out["gt_labels"][b, gi]] += int(not out["gt_ignore"][b, a, gi])
    return recs, npig


def test_micro_equals_class_aware_when_every_label_is_zero():
    thrs = oracle.iou_thresholds()
    out = _oracle(10, nc=1)
    assert (out["dets"][:, :, 5] == 0).all() and (out["gt_labels"] == 0).all()
    recs, npig = _class_aware(out, 1)
    want = oracle.accumulate_ap(recs, npig, thrs, (1, 10, 100), 1)
    got, mnpig, mrecs = micro_oracle.micro_ap([out], thrs)
    np.testing.assert_array_equal(mnpig, npig)
    assert want["map_50"] > 0.05
    for r, m in zip(recs, mrecs):
        np.testing.assert_array_equal(m["matched"], r["matched"])
        np.testing.assert_array_equal(m["ignored"], r["ignored"])
    assert got["precision"].tobytes() == want["precision"].tobytes()
    assert got["recall"].tobytes() == want["recall"].tobytes()
    assert micro_oracle.score_table(mrecs, mnpig, thrs, (1, 10, 100), 1).tobytes() == \
        micro_oracle.score_table(recs, npig, thrs, (1, 10, 100), 1).tobytes()


def _class_aware_match(out, b, thrs, nc):
    """oracle.run_pipeline's per-class COCO matching of image b: dt_match [A, T, k] (image GT index + 1), dt_ignore."""
    k, g = int(out["det_count"][b]), int(out["gt_count"][b])
    lab, gl = out["dets"][b, :k, 5].astype(np.int64), out["gt_labels"][b, :g]
    dm_all, dig_all = np.zeros((4, len(thrs), k), np.int32), np.zeros((4, len(thrs), k), np.uint8)
    for c in range(nc):
        di_, gi_ = np.nonzero(lab == c)[0], np.nonzero(gl == c)[0]
        if len(di_):
            dm, dig, _ = oracle.coco_match(out["dets"][b, di_, :4], out["gt_boxes"][b, gi_], thrs)
            dm_all[:, :, di_] = np.where(dm > 0, gi_[np.maximum(dm - 1, 0)] + 1 if len(gi_) else 0, 0)
            dig_all[:, :, di_] = dig
    return dm_all, dig_all


def test_micro_differs_where_a_wrong_class_box_overlaps_a_gt():
    """Give every third detection a wrong class: where such a box overlaps a GT it is a false positive of the
    class-aware matching and a hit of the class-agnostic one; on the untouched detections the two agree unless a
    relabelled box took the GT first."""
    thrs = oracle.iou_thresholds()
    out = _oracle(12)
    out["dets"][:, ::3, 5] = (out["dets"][:, ::3, 5] + 1) % 3
    gained = kept = 0
    for b in range(12):
        k = int(out["det_count"][b])
        _, dm, _, _ = micro_oracle.micro_records(out, b, thrs)
        ca, _ = _class_aware_match(out, b, thrs, 3)
        lab, gl = out["dets"][b, :k, 5].astype(np.int64), out["gt_labels"][b]
        for a, t, d in zip(*np.nonzero((dm > 0) & (ca == 0))):
            gained += int(d % 3 == 0 and gl[dm[a, t, d] - 1] != lab[d])
        kept += int(((ca > 0) & (dm == ca)).sum())
    assert gained > 0 and kept > 0
    recs, npig = _class_aware(out, 3)
    for b, r in enumerate(recs):
        dm, dig = _class_aware_match(out, b, thrs, 3)
        r["matched"], r["ignored"] = dm > 0, dig > 0
    mi_ap, _, _ = micro_oracle.micro_ap([out], thrs)
    ca_ap = oracle.accumulate_ap(recs, npig, thrs, (1, 10, 100), 3)
    assert mi_ap["map_50"] > ca_ap["map_50"]


def _fuzz_records(rng, n_img, K, nc, T, q):
    recs = []
    for b in range(n_img):
        k = int(rng.integers(0, K + 1))
        sc = np.sort((rng.integers(1, q + 1, k) / q).astype(np.float32))[::-1]
        recs.append(dict(labels=rng.integers(0, nc, k).astype(np.int64), scores=sc,
                         matched=rng.integers(0, 2, (4, T, k)) > 0, ignored=rng.integers(0, 4, (4, T, k)) == 0))
    return recs


SCORE_CASES = [dict(n_img=40, K=12, nc=3, T=10, max_dets=(1, 10, 100), q=8),
               dict(n_img=30, K=40, nc=5, T=10, max_dets=(1, 5, 20), q=4),
               dict(n_img=9, K=300, nc=2, T=3, max_dets=(3, 100, 300), q=64),
               dict(n_img=64, K=30, nc=1, T=16, max_dets=(100,), q=2),
               dict(n_img=3, K=4, nc=4, T=2, max_dets=(1, 2), q=3),
               dict(n_img=50, K=20, nc=3, T=10, max_dets=(1, 10, 100), q=1 << 22)]   # (nearly) continuous scores


@pytest.mark.parametrize("case", SCORE_CASES)
def test_score_table_equals_pycocotools_restatement(case):
    """Fuzzed record sets -- tied scores, ignored records in front, maxDet cuts, classes without GT or without any
    detection: the numpy score table equals the loop-for-loop pycocotools restatement exactly."""
    n_img, K, nc, T, max_dets, q = (case[k] for k in ("n_img", "K", "nc", "T", "max_dets", "q"))
    rng = np.random.default_rng(n_img * 7 + K)
    thrs = np.linspace(0.5, 0.95, T) if T > 1 else np.array([0.5])
    recs = _fuzz_records(rng, n_img, K, nc, T, q)
    if nc > 1:
        for r in recs:                                                 # a class without any detection
            r["labels"][r["labels"] == nc - 1] = 0
    for r in recs[:2]:                                                 # an ignored record at the head of class 0's sequence
        if len(r["scores"]):
            r["scores"][0], r["labels"][0], r["ignored"][:, :, 0] = 2.0, 0, True
    npig = rng.integers(1, 20, (4, nc)).astype(np.int64)
    if nc > 2:
        npig[:, 1] = 0                                                 # a class without GT
    npig[1, 0] = 0                                                     # an area range without GT
    got = micro_oracle.score_table(recs, npig, thrs, max_dets, nc)
    want = micro_oracle.pycocotools_score_table(recs, npig, thrs, max_dets, nc)
    assert got.tobytes() == want.tobytes()
    for c in range(nc):
        for a in range(4):
            if npig[a, c] == 0:
                assert (got[:, :, c, a] == -1).all()
                continue
            for mi, md in enumerate(max_dets):
                sc, _, _ = micro_oracle._sequence(recs, c, a, md)
                # recall 0 is reached at the first record of the sequence whatever its state; an empty sequence gives 0
                assert (got[:, 0, c, a, mi] == (sc[0] if len(sc) else 0.0)).all()
    assert (got > 0).any()


# ---------------------------------------------------------------------------------------------- 2-rank merge (gloo)
T = 10
MICRO_IMAGES = (3, 5)                                                 # ragged shards, the other way round from SEG_IMAGES


def _micro_shard(rank):
    """A (header, ring) pair as match_kernel leaves the class-agnostic state: one record per kept detection, label 0,
    class_rank = rank, NPIG[a][0] = non-ignored GTs of every class."""
    n, off = MICRO_IMAGES[rank], sum(MICRO_IMAGES[:rank])
    out = oracle.run_pipeline(synth.make_batch(synth.SynthConfig(batch=n, img_size=160, seed=77, image_offset=off)),
                              img_size=160, **KW)
    thrs = oracle.iou_thresholds()
    mo = dict(det_count=out["det_count"], dets=out["dets"].copy(), dt_match=np.zeros_like(out["dt_match"]),
              dt_ignore=np.zeros_like(out["dt_ignore"]))
    mo["dets"][:, :, 5] = 0
    hdr = np.zeros(HDR, np.int64)
    for b in range(n):
        _, dm, di, gi = micro_oracle.micro_records(out, b, thrs)
        k = dm.shape[2]
        mo["dt_match"][b][:, :, :k], mo["dt_ignore"][b][:, :, :k] = dm, di
        hdr[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64: 16] += (gi == 0).sum(1)
    raw = encode_records(mo, off, T)
    hdr[_lib.SWEEP_N_RECORDS], hdr[_lib.SWEEP_N_IMAGES] = len(raw), n
    ring = np.zeros((len(raw) + 5 * rank, 32), np.uint8)
    ring[:len(raw)] = raw.view(np.uint8).reshape(-1, 32)
    return hdr, ring


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
        dh, dr = _det_shard(rank)
        sh, sr, _ = _seg_shard(rank, (5, 3)[rank], (0, 5)[rank])
        mh, mr = _micro_shard(rank)
        hdrs = [torch.from_numpy(dh), torch.from_numpy(sh), torch.from_numpy(mh)]
        ns, merged = merge_sweeps(hdrs, [torch.from_numpy(dr), torch.from_numpy(sr), torch.from_numpy(mr)])
        if rank == 1:
            q.put((ns, [m.numpy().copy() for m in merged], [h.numpy().copy() for h in hdrs], calls))
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_merge_of_three_states():
    """The detection, segmentation-mAP and class-agnostic states of one DeviceSweep merge exactly as single-process
    concatenations with ONE header all-reduce and the all-gathers of the detection state alone (counts + records)."""
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_merge_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    ns, merged, hdrs, calls = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert calls == {"all_reduce": 1, "all_gather_into_tensor": 2, "other": 0}
    det = [_det_shard(r) for r in range(world)]
    seg = [_seg_shard(r, (5, 3)[r], (0, 5)[r]) for r in range(world)]
    mic = [_micro_shard(r) for r in range(world)]
    assert ns[0] == [int(h[0]) for h, _ in det] and ns[1] == [5, 3] and ns[2] == [int(h[0]) for h, _ in mic]
    assert ns[2][0] != ns[2][1]
    np.testing.assert_array_equal(merged[0], np.concatenate([r[:n] for (_, r), n in zip(det, ns[0])]))
    np.testing.assert_array_equal(merged[1], np.concatenate([s[1][:n] for s, n in zip(seg, ns[1])]))
    np.testing.assert_array_equal(merged[2], np.concatenate([r[:n] for (_, r), n in zip(mic, ns[2])]))
    np.testing.assert_array_equal(hdrs[2], mic[0][0] + mic[1][0])
    rec = decode_records(torch.from_numpy(merged[2]), T)
    assert not rec["label"].any() and (rec["class_rank"] == rec["rank"]).all()
    assert rec["image"].max() < sum(MICRO_IMAGES) and (np.diff(rec["image"].astype(np.int64)) >= 0).all()
