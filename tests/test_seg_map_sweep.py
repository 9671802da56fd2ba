"""CPU: the v3 segmentation-mAP sweep state (BtIO.seg_sweep) -- the ABI layout of the new field, its argument validation
(before any CUDA call), and the merge of a detection state and a segmentation state across a 2-rank gloo group with the
same collectives as the detection state alone."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from btpost import _lib
from btpost.sweep import HDR, decode_records, merge_sweeps
from oracle import oracle
from test_sweep import _free_port, encode_records, oracle_outputs

ROOT = Path(__file__).resolve().parents[1]


def test_btio_layout_with_seg_sweep(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "btpost.h"\nint main(){'
                   'printf("%zu %zu %zu\\n", sizeof(BtIO), offsetof(BtIO, image_base), offsetof(BtIO, seg_sweep));return 0;}')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(_lib.BtIO), _lib.BtIO.image_base.offset, _lib.BtIO.seg_sweep.offset]
    assert _lib._IO_FIELDS[-1] == "seg_sweep" and got[2] == got[0] - 8   # appended: every earlier offset is unchanged


def _params():
    p = _lib.BtParams()
    p.batch, p.num_anchors, p.nc, p.nm, p.max_det, p.max_gt = 2, 8400, 3, 32, 300, 32
    p.img_h = p.img_w = 640
    p.proto_h = p.proto_w = 160
    p.num_iou_thrs = 10
    n = C.c_size_t()
    assert _lib.load().btpost_workspace_bytes(C.byref(p), C.byref(n)) == 0
    return p, n.value


def test_seg_sweep_argument_validation_without_gpu():
    """seg_sweep needs seg_img3 and seg_prob_sum (BT_ERR_BAD_ARG) and 16-byte alignment (BT_ERR_MISALIGNED); both are
    checked before any CUDA call, by the mask stage and by btpost_run."""
    L = _lib.load()
    p, ws = _params()
    io = _lib.BtIO()
    for f in ("head", "protos", "masks_gt", "proj_weight", "dets", "det_count", "det_coeff", "det_keep", "det_anchor", "n_cand",
              "gt_count", "gt_boxes", "gt_boxes_raw", "gt_labels", "cm", "cm_pos"):
        setattr(io, f, 4096)
    masks = lambda: L.btpost_masks_parts(C.byref(p), C.byref(io), C.c_void_p(256), ws, None, _lib.MASKS_CELLS)
    run = lambda: L.btpost_run(C.byref(p), C.byref(io), C.c_void_p(256), ws, None)
    io.seg_sweep, io.seg_img3 = 8192, 4096                          # seg_prob_sum missing
    assert masks() == -1 and run() == -1
    io.seg_img3, io.seg_prob_sum = None, 4096                       # seg_img3 missing
    assert masks() == -1 and run() == -1
    io.seg_img3, io.seg_sweep = 4096, 8192 + 8                      # misaligned state
    assert masks() == -4 and run() == -4


# ---------------------------------------------------------------------------------------------- 2-rank merge (gloo)
T = 10


def _seg_shard(rank, n_images, image_offset):
    """A (header, ring) pair as finalize_kernel leaves it: one record per image, class 0, NPIG[a][0] = non-ignored GT
    masks.  Built from the oracle's per-image restatement on random (inter, |P|, |G|) triples and scores."""
    rng = np.random.default_rng(100 + rank)
    G = rng.integers(0, 12000, n_images)
    P = rng.integers(0, 12000, n_images)
    inter = np.minimum(P, G) * rng.uniform(0.3, 1.0, n_images)
    img3 = np.stack([inter.astype(np.int64), P, G], 1)
    scores = np.where(P > 0, rng.uniform(0.5, 1.0, n_images), 0.0).astype(np.float32)
    rec = oracle.seg_map_records(img3, scores, oracle.iou_thresholds())
    raw = encode_records(rec, image_offset, T)
    hdr = np.zeros(HDR, np.int64)
    hdr[_lib.SWEEP_N_RECORDS] = hdr[_lib.SWEEP_N_IMAGES] = n_images
    hdr[_lib.SWEEP_NPIG: _lib.SWEEP_NPIG + 64: 16] = (1 - rec["gt_ignore"][:, :, 0]).sum(0)
    ring = np.zeros((n_images + 3 * rank, 32), np.uint8)            # rings of different capacity per rank
    ring[:n_images] = raw.view(np.uint8).reshape(-1, 32)
    return hdr, ring, raw


SEG_IMAGES = (5, 3)                                                  # ragged shards: 5 images on rank 0, 3 on rank 1


def _det_shard(rank):
    out, _ = oracle_outputs(4, image_offset=4 * rank)
    raw = encode_records(out, 4 * rank)
    hdr = np.zeros(HDR, np.int64)
    hdr[_lib.SWEEP_N_RECORDS], hdr[_lib.SWEEP_N_IMAGES] = len(raw), 4
    ring = np.zeros((len(raw) + 11 * (1 - rank), 32), np.uint8)
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
        sh, sr, _ = _seg_shard(rank, SEG_IMAGES[rank], sum(SEG_IMAGES[:rank]))
        hdrs = [torch.from_numpy(dh), torch.from_numpy(sh)]
        ns, merged = merge_sweeps(hdrs, [torch.from_numpy(dr), torch.from_numpy(sr)])
        if rank == 1:
            q.put((ns, [m.numpy().copy() for m in merged], [h.numpy().copy() for h in hdrs], calls))
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_merge_of_detection_and_segmentation_states():
    """Both states of a DeviceSweep with a segmentation ring merge exactly as single-process concatenations, with ONE
    header all-reduce and the two all-gathers of the detection state alone."""
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
    seg = [_seg_shard(r, SEG_IMAGES[r], sum(SEG_IMAGES[:r])) for r in range(world)]
    assert ns == [[int(h[0]) for h, _ in det], list(SEG_IMAGES)]
    np.testing.assert_array_equal(merged[0], np.concatenate([r[:n] for (_, r), n in zip(det, ns[0])]))
    np.testing.assert_array_equal(merged[1], np.concatenate([s[1][:n] for s, n in zip(seg, SEG_IMAGES)]))
    np.testing.assert_array_equal(hdrs[0], det[0][0] + det[1][0])
    np.testing.assert_array_equal(hdrs[1], seg[0][0] + seg[1][0])
    rec = decode_records(torch.from_numpy(merged[1]), T)
    np.testing.assert_array_equal(rec["image"], np.arange(sum(SEG_IMAGES)))
    assert not rec["label"].any() and not rec["rank"].any() and not rec["class_rank"].any()
