"""A float64 restatement of the reference's statements, written with torch and independent of the oracle.

The oracle (oracle/btpost_oracle.c) restates the kernels' fp32 rounding on purpose, so a mistake shared by both
would pass a bit-exact comparison.  The functions here take the INPUTS of a batch and the OUTPUTS of either the
CUDA library or the oracle, recompute what the reference computes in float64, and check the outputs against it:
exactly where the fp32 result is determined (box decode, labels, scores, coefficients), and within a bound derived
from the number of fp32 roundings everywhere else.

Rounding bounds.  u = 2^-24 (unit roundoff of fp32).  A projector logit is `bias + sum_k w_k p_k` over nm = 32
channels, evaluated as 32 chained fused multiply-adds: <= 32 roundings, and the classical bound for recursive
summation gives |err| <= gamma_32 * (|b| + sum_k |w_k||p_k|), gamma_n = n u / (1 - n u).  The bilinear x4 upsample
(align_corners=False, S = 4 PW) has exact weights in {0, 1/8, 3/8, 5/8, 7/8, 1}, and each corner value passes through
at most 4 more roundings (`fma(h0, fma(w0, v00, w1 * v01), h1 * fma(w0, v10, w1 * v11))`); the weights are
non-negative and sum to 1, so the upsampled bound is the bilinear upsample of the prototype-resolution bound with
36 roundings.  C_ROUND = 37 adds one unit for gamma_36's second-order term (36 u < 3e-6) and the float64
evaluation of the reference itself (< 40 * 2^-53 relative).  Instance logits are the same with bias 0.

The fp32 threshold `sigmoid(x) > 0.5` holds exactly for x > 1.5 u (tests/test_oracle_pinning.py), so a pixel is
certain only where the float64 logit is below -E or above E + 1.5 u; the pixels in between form the band.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

U = 2.0 ** -24
C_ROUND = 37
SIGMOID_HALF_X = 1.5 * 2.0 ** -24
EPS = 1e-7                                     # the reference's Dice / IoU epsilon (src/test_model.py:15-23)


def _f64(a):
    return torch.from_numpy(np.ascontiguousarray(a)).double()


def _up(x, S):
    """F.interpolate(bilinear, align_corners=False) of [..., PH, PW] to [..., S, S] in float64."""
    lead = x.shape[:-2]
    y = F.interpolate(x.reshape(-1, 1, *x.shape[-2:]), size=(S, S), mode="bilinear", align_corners=False)
    return y.reshape(*lead, S, S)


# ------------------------------------------------------------------------------------------------- detections
def check_l2_detections(head, out, nc, S, conf=0.05, clamp=True):
    """Every kept detection against its anchor's column of the L2 head (Ultralytics xywh2xyxy, then the filter's
    clamp; label = first argmax over the nc class rows, score = that row's value).  x1 = cx - w/2 is exact in float64
    for fp32 operands, so rounding it once to fp32 gives the kernel's value bit for bit.  Returns the kept labels."""
    labels = []
    for b in range(head.shape[0]):
        k = int(out["det_count"][b])
        a = out["det_anchor"][b, :k].astype(np.int64)
        col = head[b][:, a].astype(np.float64)
        cx, cy, w, h = col[0], col[1], col[2], col[3]
        box = np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1).astype(np.float32)
        if clamp:
            box = np.clip(box, np.float32(0), np.float32(S))
        assert out["dets"][b, :k, :4].tobytes() == box.tobytes(), f"boxes of image {b}"
        sc = col[4:4 + nc]
        lab = np.argmax(sc, 0)                                               # first maximum
        np.testing.assert_array_equal(out["dets"][b, :k, 5], lab.astype(np.float32), err_msg=f"labels of image {b}")
        np.testing.assert_array_equal(out["dets"][b, :k, 4], sc.max(0).astype(np.float32), err_msg=f"scores of image {b}")
        assert np.all(out["dets"][b, :k, 4] > conf)
        assert out["det_coeff"][b, :k].tobytes() == np.ascontiguousarray(head[b][4 + nc:, a].T).tobytes()
        labels.append(lab)
    return np.concatenate(labels) if labels else np.zeros(0, np.int64)


def l1_decode(maps_img, S, nc, R=16):
    """running_main_v2.py:743-775 in float64 for one image: DFL softmax expectation over R bins, anchors (x+.5, y+.5),
    stride S / W.  Returns (boxes [N, 4] xyxy, class logits [N, nc])."""
    boxes, logits = [], []
    for m in maps_img:
        t = _f64(m)
        _, H, W = t.shape
        st = S / W
        dfl = torch.softmax(t[:4 * R].reshape(4, R, H * W), 1)
        d = (dfl * torch.arange(R, dtype=torch.float64)[None, :, None]).sum(1) * st      # [4, HW] ltrb in pixels
        gy, gx = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64), indexing="ij")
        ax, ay = (gx.reshape(-1) + 0.5) * st, (gy.reshape(-1) + 0.5) * st
        boxes.append(torch.stack([ax - d[0], ay - d[1], ax + d[2], ay + d[3]], 1))
        logits.append(t[4 * R:].reshape(nc, H * W).T)
    return torch.cat(boxes).numpy(), torch.cat(logits).numpy()


def check_l1_detections(maps, coeffs, out, nc, S, R=16, clamp=True):
    """Kept detections of the raw-map layout against the float64 DFL decode: boxes within the atol = 1e-4 that pins
    the oracle's fma-polynomial exp against torch (tests/test_oracle_pinning.py), scores = sigmoid of the label's
    logit within 3e-6 relative, the label a maximum of the logits up to the fp32 sigmoid's rounding.  Returns the
    kept labels."""
    labels = []
    for b in range(maps[0].shape[0]):
        boxes, logits = l1_decode([m[b] for m in maps], S, nc, R)
        k = int(out["det_count"][b])
        a = out["det_anchor"][b, :k].astype(np.int64)
        box = np.clip(boxes[a], 0, S) if clamp else boxes[a]
        np.testing.assert_allclose(out["dets"][b, :k, :4], box, rtol=0, atol=1e-4, err_msg=f"boxes of image {b}")
        lab = out["dets"][b, :k, 5].astype(np.int64)
        lg = logits[a]
        chosen = lg[np.arange(k), lab]
        assert np.all(chosen >= lg.max(1) - 1e-5 * np.maximum(1.0, np.abs(lg.max(1)))), f"labels of image {b}"
        np.testing.assert_allclose(out["dets"][b, :k, 4], 1.0 / (1.0 + np.exp(-chosen)), rtol=3e-6, atol=0)
        assert out["det_coeff"][b, :k].tobytes() == np.ascontiguousarray(coeffs[b][:, a].T).tobytes()
        labels.append(lab)
    return np.concatenate(labels) if labels else np.zeros(0, np.int64)


# ------------------------------------------------------------------------------------------------- projector
def projector(protos, weight, bias, S):
    """Conv2d(nm -> 1, k=1) + bilinear to S (running_main_v2.py:689-699) in float64, and the per-pixel rounding bound E
    of the module docstring.  Returns (logits [B, S, S], E [B, S, S])."""
    p, w = _f64(protos), _f64(weight)
    lg = float(bias) + torch.einsum("k,bkhw->bhw", w, p)
    mag = abs(float(bias)) + torch.einsum("k,bkhw->bhw", w.abs(), p.abs())
    return _up(lg, S), C_ROUND * U * _up(mag, S)


def band(ref, E):
    """Pixels whose fp32 threshold the bound cannot decide.  Where E = 0 (outside a crop box) the logit is exactly 0."""
    return (E > 0) & (ref >= -E) & (ref <= E + SIGMOID_HALF_X)


def check_projector(protos, weight, bias, masks_gt, out, S):
    """seg_logits within E of the float64 logits; seg_mask = ref > 0 outside the band; seg_img3 / seg_dice / seg_iou
    within what the band leaves open.  Returns (the float64 logits and E, for soft Dice, and the band's pixel count)."""
    ref, E = projector(protos, weight, bias, S)
    got = torch.from_numpy(out["seg_logits"]).double()
    over = (got - ref).abs() - E
    assert float(over.max()) <= 0, f"seg_logits off the float64 reference by {float(over.max())} beyond the bound"
    bd = band(ref, E)
    sure = (ref > E + SIGMOID_HALF_X)
    mask = torch.from_numpy(out["seg_mask"].astype(bool))
    assert bool((mask[~bd] == sure[~bd]).all()), "seg_mask differs from the float64 reference outside the band"
    gt = torch.from_numpy(np.ascontiguousarray(masks_gt[:, 0]) != 0)
    check_dice_iou(sure, bd, gt, out["seg_img3"], out["seg_dice"], out["seg_iou"])
    return ref, E, int(bd.sum())


def check_dice_iou(sure, bd, gt, img3, dice, iou):
    """Dice and IoU are increasing in the foreground pixels inside the GT mask and decreasing in those outside it, so
    the kernel's values lie between the band's best and worst assignment (reference epsilon 1e-7), widened by 1e-5."""
    for b in range(sure.shape[0]):
        g = gt[b]
        I0, P0, G = int((sure[b] & g).sum()), int(sure[b].sum()), int(g.sum())
        b_in, b_out = int((bd[b] & g).sum()), int((bd[b] & ~g).sum())
        assert img3[b, 2] == G and I0 <= img3[b, 0] <= I0 + b_in and P0 <= img3[b, 1] <= P0 + b_in + b_out, f"image {b}"
        d = lambda I, P: (2.0 * I + EPS) / (P + G + EPS)
        j = lambda I, P: (I + EPS) / (P + G - I + EPS)
        for name, f, v in (("dice", d, dice[b]), ("iou", j, iou[b])):
            lo, hi = f(I0, P0 + b_out), f(I0 + b_in, P0 + b_in)
            assert lo * (1 - 1e-5) <= float(v) <= hi * (1 + 1e-5), f"seg_{name} of image {b}: {v} not in [{lo}, {hi}]"


def check_soft_dice(ref, E, masks_gt, soft_dice):
    """v3's soft Dice (SURVEY.md A.4): 2 sum(sigmoid(x) t) / (sum sigmoid(x) + sum t) on the float64 logits.  Per pixel
    the kernel's probability differs from sigmoid(ref) by at most E / 4 (sigmoid' <= 1/4), 8 u for its fp32 sigmoid
    (the fma-polynomial exp within 2 ulp of libm's, libm's within 1 ulp, one addition, one division; p <= 1; the 2 ulp
    are measured on [-88, 0] and taken here for the arguments of either sign) and 2^-41 for the rounding
    to 2^-40 fixed point; summed over the pixels that bounds A and P, and the fp32 result adds 2^-24 relative."""
    p = torch.sigmoid(ref)
    t = torch.from_numpy(np.ascontiguousarray(masks_gt[:, 0]) != 0).double()
    d = E / 4 + 8 * U + 2.0 ** -41
    for b in range(ref.shape[0]):
        A, P, G = float((p[b] * t[b]).sum()), float(p[b].sum()), float(t[b].sum())
        dA, dP = float((d[b] * t[b]).sum()), float(d[b].sum())
        lo, hi = 2 * (A - dA) / (P + dP + G), 2 * (A + dA) / (P - dP + G)
        v = float(soft_dice[b])
        assert lo * (1 - 2 * U) <= v <= hi * (1 + 2 * U), f"seg_soft_dice of image {b}: {v} not in [{lo}, {hi}]"


# ------------------------------------------------------------------------------------------------- instance masks
def check_instances(protos, out, planes_of, S, crop=True, chunk=32):
    """Every kept detection's mask (src/test_model.py:80-85 with the Ultralytics crop): coefficients . prototypes in
    float64, crop at prototype resolution (keep r >= y1 PH/S, r < y2 PH/S, same for the columns with PW), bilinear to S,
    > 0.  `planes_of(b)` gives image b's [det_count, S, S] masks; they must agree outside the band.  Returns the band's
    pixel count over all detections."""
    n_band = 0
    for b in range(protos.shape[0]):
        k = int(out["det_count"][b])
        planes = torch.from_numpy(np.ascontiguousarray(planes_of(b)).astype(bool))
        assert planes.shape[0] == k
        p = _f64(protos[b])
        _, PH, PW = p.shape
        r = torch.arange(PH, dtype=torch.float64)[:, None]
        c = torch.arange(PW, dtype=torch.float64)[None, :]
        for i0 in range(0, k, chunk):
            i1 = min(k, i0 + chunk)
            co = _f64(out["det_coeff"][b, i0:i1])
            lg = torch.einsum("qk,khw->qhw", co, p)
            mag = torch.einsum("qk,khw->qhw", co.abs(), p.abs())
            if crop:
                bx = _f64(out["dets"][b, i0:i1, :4])
                x1, y1, x2, y2 = (bx[:, j, None, None] for j in range(4))
                keep = ((c >= x1 * PW / S) & (c < x2 * PW / S) & (r >= y1 * PH / S) & (r < y2 * PH / S)).double()
                lg, mag = lg * keep, mag * keep
            ref, E = _up(lg, S), C_ROUND * U * _up(mag, S)
            bd = band(ref, E)
            sure = ref > E + SIGMOID_HALF_X
            bad = (planes[i0:i1] != sure) & ~bd
            assert not bool(bad.any()), (f"image {b}: instance masks {sorted(set((i0 + bad.nonzero()[:, 0]).tolist()))[:8]} "
                                         "differ from the float64 reference outside the band")
            n_band += int(bd.sum())
    return n_band
