"""CPU: surface distances of the projector mask (btpost_surface_distance) -- the scipy restatement of tests/surface_oracle.py
against an independent brute-force one (minimum over edge-pixel pairs, the quantile formula written out on the sorted
integer squared distances), the arguments both entry points reject before any CUDA call, and the fixed-point bounds."""
import ctypes as C
import math

import numpy as np
import pytest

import surface_oracle as so
from btpost import _lib


def brute_edges(m):
    """A foreground pixel is an edge pixel unless its four neighbours are all foreground (outside = background)."""
    m = np.asarray(m) != 0
    p = np.pad(m, 1)
    inner = p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:]
    return m & ~inner


def brute_quantile95(d2_sorted):
    n = len(d2_sorted)
    rank = 0.95 * (n - 1)
    lo, hi = math.floor(rank), math.ceil(rank)
    a, b, w = math.sqrt(float(d2_sorted[lo])), math.sqrt(float(d2_sorted[hi])), rank - lo
    return a + w * (b - a) if w < 0.5 else b - (b - a) * (1 - w)


def brute(pred, gt):
    ep, eg = np.argwhere(brute_edges(pred)), np.argwhere(brute_edges(gt))
    if len(ep) == 0 or len(eg) == 0:
        return float("nan"), float("nan"), float("nan")
    d2 = ((ep[:, None, :] - eg[None, :, :]) ** 2).sum(-1)          # integer squared distances, every pair
    a, b = np.sort(d2.min(1)), np.sort(d2.min(0))
    hd = math.sqrt(float(max(a[-1], b[-1])))
    hd95 = max(brute_quantile95(a), brute_quantile95(b))
    assd = float(np.sqrt(np.concatenate([a, b]).astype(np.float64)).mean())
    return hd, hd95, assd


def mask_zoo(rng, S):
    """Random masks, and the shapes the kernel's edge cases come from."""
    yy, xx = np.mgrid[:S, :S]
    z = np.zeros((S, S), bool)
    one = z.copy()
    one[rng.integers(S), rng.integers(S)] = True
    line = z.copy()
    line[rng.integers(S)] = True
    col = z.copy()
    col[:, rng.integers(S)] = True
    blob = (yy - rng.integers(S)) ** 2 + (xx - rng.integers(S)) ** 2 < rng.integers(1, S * S)
    border = z.copy()
    border[: rng.integers(1, S + 1), : rng.integers(1, S + 1)] = True           # touches the top and left borders
    return [rng.random((S, S)) < rng.uniform(0.02, 0.9), (yy + xx) % 2 == 0, np.ones((S, S), bool), z, one, line, col,
            blob, border, blob | one]


def cases(seed=5, count=300):
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < count:
        S = int(rng.choice([2, 3, 7, 16, 23, 32]))
        zoo = mask_zoo(rng, S)
        a, b = zoo[rng.integers(len(zoo))], zoo[rng.integers(len(zoo))]
        out.append((a, b))
        if len(out) % 25 == 0:
            out.append((a, a.copy()))                                   # identical pair: every distance 0
    return out


def test_oracle_equals_brute_force():
    """hd and hd95 equal (double), assd within 1e-12 relative (a different summation order), NaN together; the cases
    cover n = 1 and edge counts n for which 0.95 (n - 1) is an integer."""
    seen_n = set()
    for pred, gt in cases():
        got, want = so.surface_distance(pred, gt), brute(pred, gt)
        if np.isnan(want[0]):
            assert all(np.isnan(v) for v in got), (pred, gt)
            continue
        assert got[0] == want[0] and got[1] == want[1], (got, want)
        assert got[2] == pytest.approx(want[2], rel=1e-12, abs=0.0)
        seen_n.update(int(brute_edges(m).sum()) for m in (pred, gt))
    assert 1 in seen_n and any(n > 1 and (19 * (n - 1)) % 20 == 0 for n in seen_n)


def test_oracle_batch_and_accumulator():
    rng = np.random.default_rng(9)
    S = 24
    pred = np.stack([mask_zoo(rng, S)[i] for i in (0, 1, 3, 4, 7)]).astype(np.uint8)   # image 2 empty
    gt = np.stack([mask_zoo(rng, S)[i] for i in (7, 0, 7, 3, 4)]).astype(np.float32)[:, None]   # image 3 empty
    hd, hd95, assd = so.surface_batch(pred, gt)
    assert hd.dtype == np.float32 and np.isnan(hd[[2, 3]]).all() and np.isfinite(hd[[0, 1, 4]]).all()
    for b in (0, 1, 4):
        want = brute(pred[b], gt[b, 0])
        assert hd[b] == np.float32(want[0]) and hd95[b] == np.float32(want[1])
    acc = so.accumulate(hd, hd95, assd)
    assert acc[3] == 3 and acc[0] == sum(int(np.rint(float(hd[b]) * 2.0 ** 32)) for b in (0, 1, 4))
    m = so.means(acc)
    assert m[0] == pytest.approx(float(np.nanmean(hd.astype(np.float64))), rel=1e-12)
    assert all(np.isnan(v) for v in so.means(np.zeros(4, np.int64)))


def test_fixed_point_bounds():
    """The kernel sums round(d * 2^30) as int64 over both directions of an image: with every pixel of a 1280^2 image an
    edge pixel of both masks and every distance at its largest (the diagonal), the sum stays below 2^63.  The accumulator
    words (2^32 units, values below 2^11) hold more than a million images."""
    S = 1280
    d_max = math.sqrt(2.0) * (S - 1)
    assert 2 * S * S * round(d_max * 2.0 ** 30) < 2 ** 63
    assert 2 * (S - 1) ** 2 < 2 ** 22                                     # squared distances fit the 22-bit select
    assert (1 << 20) * round(d_max * 2.0 ** 32) < 2 ** 63


def test_surface_argument_validation_without_gpu():
    """Every error of btpost_surface_bytes / btpost_surface_distance is returned before any CUDA call (fake pointers)."""
    L = _lib.load()
    n = C.c_size_t()
    assert L.btpost_surface_bytes(2, 640, None) == -1
    assert L.btpost_surface_bytes(0, 640, C.byref(n)) == -1
    assert L.btpost_surface_bytes(2, 0, C.byref(n)) == -1
    assert L.btpost_surface_bytes(2, 650, C.byref(n)) == -2                      # not a multiple of 32
    assert L.btpost_surface_bytes(2, 1312, C.byref(n)) == -2                     # above 1280
    assert L.btpost_surface_bytes(2, 1280, C.byref(n)) == 0 and n.value >= 8 * 2 * 1280 * 1280
    assert L.btpost_surface_bytes(64, 640, C.byref(n)) == 0 and n.value == 8 * 64 * 640 * 640 + 4096
    B, S = 2, 640
    assert L.btpost_surface_bytes(B, S, C.byref(n)) == 0
    ws = n.value
    good = dict(batch=B, img=S, pred=4096, gt=8192, dt=_lib.MASK_U8, hd=12288, hd95=16384, assd=20480, acc=None,
                scratch=1 << 20, nbytes=ws)

    def call(**kw):
        a = dict(good, **kw)
        return L.btpost_surface_distance(a["batch"], a["img"], a["pred"], a["gt"], a["dt"], a["hd"], a["hd95"], a["assd"],
                                         a["acc"], a["scratch"], a["nbytes"], None)
    for k in ("pred", "gt", "hd", "hd95", "assd", "scratch"):
        assert call(**{k: None}) == -1, k
    assert call(batch=0) == -1 and call(batch=-3) == -1 and call(img=0) == -1
    assert call(dt=2) == -1 and call(dt=-1) == -1
    assert call(img=656) == -2 and call(img=1312) == -2
    assert call(pred=4104) == -4 and call(gt=8200) == -4 and call(scratch=(1 << 20) + 128) == -4
    assert call(nbytes=ws - 1) == -3
    assert call(img=1280, nbytes=ws) == -3                                       # the scratch is sized for the shape
    assert b"workspace" in L.btpost_error_string(-3)
