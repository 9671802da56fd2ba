"""-m gpu: surface distances of the projector mask (btpost_surface_distance, PostConfig.with_surface_dist,
DeviceSweep(surface=True)) against the scipy restatement of tests/surface_oracle.py: hd and hd95 bit for bit, assd within
one fp32 ulp, the accumulator words exactly; through the entry point alone, PostProcessor and Pipeline's captured steps."""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers
import surface_oracle as so
from btpost import Pipeline, PostConfig, PostProcessor, _lib
from btpost.sweep import DeviceSweep
from oracle import oracle
from test_gpu_seg_map_sweep import seg_batch

pytestmark = pytest.mark.gpu

THRS = oracle.iou_thresholds()
MAX_DETS = (1, 10, 100)
SURF_KEYS = ("seg_hd", "seg_hd95", "seg_assd", "seg_surf_acc")


def projector_like(rng, S):
    """Upsampled noise, thresholded: ragged blobs with dense edges, like the synthetic projector's mask."""
    lo = torch.from_numpy(rng.standard_normal((1, 1, S // 16, S // 16)).astype(np.float32))
    return (torch.nn.functional.interpolate(lo, size=(S, S), mode="bilinear")[0, 0] > 0.3).numpy()


def ellipses(rng, S, n):
    yy, xx = np.mgrid[:S, :S].astype(np.float64)
    m = np.zeros((S, S), bool)
    for _ in range(n):
        cy, cx, ry, rx = rng.uniform(0, S), rng.uniform(0, S), rng.uniform(2, S / 4), rng.uniform(2, S / 4)
        m |= ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1.0
    return m


def mask_pairs(B, S, seed):
    """B (pred, gt) pairs that cycle through: projector-like blobs against ellipse unions, salt-and-pepper noise, a
    checkerboard (every foreground pixel an edge pixel), a full mask, single pixels far apart, 1-pixel lines,
    border-touching rectangles, an identical pair (every distance 0), one empty mask and two empty masks."""
    rng = np.random.default_rng(seed)
    z = np.zeros((S, S), bool)
    yy, xx = np.mgrid[:S, :S]

    def point(y, x):
        m = z.copy()
        m[y, x] = True
        return m

    def line(r=None, c=None):
        m = z.copy()
        if r is not None:
            m[r] = True
        else:
            m[:, c] = True
        return m

    def rect(y0, y1, x0, x1):
        m = z.copy()
        m[y0:y1, x0:x1] = True
        return m
    kinds = [
        lambda: (projector_like(rng, S), ellipses(rng, S, 3)),
        lambda: (projector_like(rng, S), projector_like(rng, S)),
        lambda: (rng.random((S, S)) < 0.3, ellipses(rng, S, 2)),
        lambda: ((yy + xx) % 2 == 0, ellipses(rng, S, 1)),
        lambda: (np.ones((S, S), bool), projector_like(rng, S)),
        lambda: (point(0, 0), point(S - 1, S - 1)),
        lambda: (line(r=int(rng.integers(S))), line(c=int(rng.integers(S)))),
        lambda: (rect(0, S // 3, 0, S), rect(S // 2, S, S - S // 5, S)),
        lambda: (lambda m: (m, m.copy()))(ellipses(rng, S, 4)),
        lambda: (z.copy(), ellipses(rng, S, 2)),
        lambda: (projector_like(rng, S), z.copy()),
        lambda: (z.copy(), z.copy()),
        lambda: ((yy + xx) % 2 == 0, point(S // 2, S // 3)),
    ]
    pairs = [kinds[b % len(kinds)]() for b in range(B)]
    return np.stack([p for p, _ in pairs]).astype(np.uint8), np.stack([g for _, g in pairs]).astype(np.uint8)


_oracle_cache = {}


def oracle_for(B, S, seed):
    key = (B, S, seed)
    if key not in _oracle_cache:
        pred, gt = mask_pairs(B, S, seed)
        _oracle_cache[key] = (pred, gt, so.surface_batch(pred, gt))
    return _oracle_cache[key]


def surface(pred, gt, acc=None):
    """btpost_surface_distance on device tensors; returns (hd, hd95, assd) device tensors."""
    L = _lib.load()
    B, S = pred.shape[0], pred.shape[-1]
    n = C.c_size_t()
    _lib.check(L.btpost_surface_bytes(B, S, C.byref(n)), "btpost_surface_bytes")
    scratch = torch.empty(n.value, dtype=torch.uint8, device=pred.device)
    out = [torch.empty(B, dtype=torch.float32, device=pred.device) for _ in range(3)]
    dt = _lib.MASK_F32 if gt.dtype == torch.float32 else _lib.MASK_U8
    rc = L.btpost_surface_distance(B, S, C.c_void_p(pred.data_ptr()), C.c_void_p(gt.data_ptr()), dt,
                                   *(C.c_void_p(t.data_ptr()) for t in out), C.c_void_p(acc.data_ptr() if acc is not None else 0),
                                   C.c_void_p(scratch.data_ptr()), C.c_size_t(n.value),
                                   C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "btpost_surface_distance")
    return out


def assert_equals_oracle(got, want):
    hd, hd95, assd = (t.cpu().numpy() if isinstance(t, torch.Tensor) else t for t in got)
    np.testing.assert_array_equal(hd, want[0])                  # fp32, NaN where undefined
    np.testing.assert_array_equal(hd95, want[1])
    np.testing.assert_array_equal(np.isnan(assd), np.isnan(want[2]))
    ok = ~np.isnan(want[2])
    assert (np.abs(assd[ok].astype(np.float64) - want[2][ok]) <= np.spacing(want[2][ok]).astype(np.float64)).all()


@pytest.mark.parametrize("gt_f32", [False, True])
@pytest.mark.parametrize("S", [160, 640, 1024])
def test_entry_point_equals_oracle(S, gt_f32):
    B = 13
    pred, gt, want = oracle_for(B, S, 40 + S)
    assert np.isnan(want[0]).sum() == 3 and (want[0][~np.isnan(want[0])] > 0).any() and (want[0] == 0).any()
    dp = torch.from_numpy(pred).cuda()
    dg = torch.from_numpy(gt[:, None].astype(np.float32) if gt_f32 else gt[:, None]).cuda()
    acc = torch.zeros(4, dtype=torch.int64, device="cuda")
    first = surface(dp, dg, acc)
    torch.cuda.synchronize()
    assert_equals_oracle(first, want)
    words = so.accumulate(*want)
    np.testing.assert_array_equal(acc.cpu().numpy(), words)
    second = surface(dp, dg, acc)                               # same bytes again; acc adds the same words once more
    torch.cuda.synchronize()
    for a, b in zip(first, second):
        assert a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()
    np.testing.assert_array_equal(acc.cpu().numpy(), 2 * words)
    sub = surface(dp[3:9].contiguous(), dg[3:9].contiguous())    # another batch composition: the same per-image bytes
    torch.cuda.synchronize()
    for a, b in zip(first, sub):
        assert a[3:9].cpu().numpy().tobytes() == b.cpu().numpy().tobytes()


def test_entry_point_batch_of_64_at_640():
    B, S = 64, 640
    pred, gt, want = oracle_for(B, S, 7)
    acc = torch.zeros(4, dtype=torch.int64, device="cuda")
    got = surface(torch.from_numpy(pred).cuda(), torch.from_numpy(gt[:, None]).cuda(), acc)
    torch.cuda.synchronize()
    assert_equals_oracle(got, want)
    np.testing.assert_array_equal(acc.cpu().numpy(), so.accumulate(*want))


def cfg_for(B, S, **kw):
    return PostConfig(batch=B, img_size=S, max_det=20, gt_mode=1, with_coco=True, **kw)


def run(pp, batch):
    d = helpers.to_dev(batch, "cuda:0")
    out = pp.run(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"], d["proj_weight"], d["proj_bias"])
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def oracle_seg_mask(batch, S):
    return np.stack([oracle.threshold(oracle.project_upsample(batch["protos"][b], batch["proj_weight"], batch["proj_bias"], S)[1])
                     for b in range(batch["protos"].shape[0])])


@pytest.mark.parametrize("S", [160, 640])
def test_post_processor_equals_oracle_and_leaves_other_outputs_unchanged(S):
    B = 4 if S == 160 else 3
    batch = seg_batch(B, S, 500 + S)
    got = run(PostProcessor(cfg_for(B, S, with_surface_dist=True), "cuda:0"), batch)
    base = run(PostProcessor(cfg_for(B, S, with_seg_mask=True), "cuda:0"), batch)
    np.testing.assert_array_equal(got["seg_mask"], oracle_seg_mask(batch, S))
    want = so.surface_batch(got["seg_mask"], batch["masks_gt"])
    assert_equals_oracle((got["seg_hd"], got["seg_hd95"], got["seg_assd"]), want)
    np.testing.assert_array_equal(got["seg_surf_acc"], so.accumulate(*want))
    assert set(got) == set(base) | set(SURF_KEYS)
    for k, v in base.items():
        assert got[k].tobytes() == v.tobytes(), k              # bit for bit, floats too


def test_pipeline_and_device_sweep():
    """Captured Pipeline steps (auto_image_offset) add every image into the sweep's seg_surf_acc: finish() returns the
    restatement's means over the images with defined values, and the accumulator words do not depend on the pipeline depth
    (nor on whether they live in a sweep header or in Pipeline.shared)."""
    B, S, nb = 4, 160, 6
    batches = [seg_batch(B, S, 91, image_offset=B * i) for i in range(nb)]
    for b in batches[1:3]:                                      # empty GT masks: undefined, not counted
        b["masks_gt"][0] = 0
    want = [so.surface_batch(oracle_seg_mask(b, S), b["masks_gt"]) for b in batches]
    want = tuple(np.concatenate([w[i] for w in want]) for i in range(3))
    words = so.accumulate(*want)
    assert 0 < words[3] < nb * B
    w = helpers.to_dev(batches[0], "cuda:0")["proj_weight"]
    got = {}
    for depth, use_sweep in ((2, True), (3, True), (2, False)):
        sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=nb * B * 20, max_det_per_image=20, device="cuda:0",
                            surface=True) if use_sweep else None
        pipe = Pipeline(cfg_for(B, S, with_surface_dist=True), "cuda:0", depth=depth, proj_weight=w, sweep=sweep,
                        auto_image_offset=True)
        for b in batches:
            d = helpers.to_dev(b, "cuda:0")
            pipe.submit(d["head"], d["protos"], d["det_boxes_gt"], d["masks_gt"])
        pipe.join()
        torch.cuda.synchronize()
        got[(depth, use_sweep)] = pipe.counters("seg_surf_acc").cpu().numpy().copy()
        if use_sweep:
            res = sweep.finish()
            assert res["n_surface_images"] == words[3] and res["n_images"] == nb * B
            assert (res["seg_hd"], res["seg_hd95"], res["seg_assd"]) == so.means(words)
    for v in got.values():
        np.testing.assert_array_equal(v, words)


def test_surface_sweep_needs_with_surface_dist():
    sweep = DeviceSweep(3, THRS, MAX_DETS, capacity=4096, max_det_per_image=20, device="cuda:0", surface=True)
    with pytest.raises(ValueError, match="with_surface_dist"):
        PostProcessor(cfg_for(4, 160), "cuda:0", sweep=sweep)
    PostProcessor(cfg_for(4, 160, with_surface_dist=True), "cuda:0", sweep=sweep)
    res = sweep.finish()
    assert res["n_surface_images"] == 0 and np.isnan(res["seg_hd"])
