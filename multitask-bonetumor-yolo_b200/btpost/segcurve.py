"""Binned precision-recall and ROC curves of the projector probabilities (torchmetrics' `BinaryPrecisionRecallCurve`,
`BinaryROC`, `BinaryAUROC` and `BinaryAveragePrecision` with ``thresholds=T``; DESIGN.md §4).

`btpost_seg_curve` leaves ``hist [2, T+1]`` int64 on the device: ``hist[t][j]`` = pixels with GT bit t and exactly j
thresholds <= p.  This module is the one place that turns it into torchmetrics' state and curves: the thresholds of an
int or a list, ``hist -> confmat [T, 2, 2]`` ([threshold, target, pred], torchmetrics' own layout) and the curves, AP
and AUROC, computed in float64 from the exact counts (torchmetrics computes them in fp32, which rounds counts above
2^24)."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

MAX_THRESHOLDS = _lib.BT_MAX_CURVE_THRS


def thresholds(spec) -> np.ndarray:
    """fp32 thresholds of ``spec``: an int T is ``torch.linspace(0, 1, T)`` in fp32 (what torchmetrics builds), a list
    (or array) is taken as fp32 values.  2 <= T <= 1024, every value in [0, 1], non-decreasing; ValueError otherwise."""
    if isinstance(spec, (int, np.integer)) and not isinstance(spec, bool):
        if not 2 <= int(spec) <= MAX_THRESHOLDS:
            raise ValueError(f"seg_curve: T must be in 2 .. {MAX_THRESHOLDS}, got {int(spec)}")
        return torch.linspace(0, 1, int(spec), dtype=torch.float32).numpy()
    thr = np.asarray(spec, dtype=np.float32).reshape(-1)
    if not 2 <= thr.size <= MAX_THRESHOLDS:
        raise ValueError(f"seg_curve: between 2 and {MAX_THRESHOLDS} thresholds, got {thr.size}")
    if not ((thr >= 0) & (thr <= 1)).all():
        raise ValueError("seg_curve: thresholds must lie in [0, 1] (and not be NaN)")
    if (np.diff(thr) < 0).any():
        raise ValueError("seg_curve: thresholds must be non-decreasing")
    return thr


def confmat(hist) -> np.ndarray:
    """``hist [2, T+1]`` -> int64 ``[T, 2, 2]`` indexed [threshold k, target, pred]: pred = 1 are the pixels with more
    than k thresholds <= p, i.e. p >= thr[k]."""
    h = np.asarray(hist.cpu() if isinstance(hist, torch.Tensor) else hist, dtype=np.int64)
    T = h.shape[1] - 1
    above = np.cumsum(h[:, ::-1], axis=1)[:, ::-1][:, 1:]     # above[t][k] = sum_{j > k} hist[t][j]
    below = h.sum(1, keepdims=True) - above
    cm = np.empty((T, 2, 2), np.int64)
    cm[:, :, 1] = above.T
    cm[:, :, 0] = below.T
    return cm


def _div(num, den, zero):
    num, den = np.asarray(num, np.float64), np.asarray(den, np.float64)
    out = np.full(num.shape, float(zero))
    np.divide(num, den, out=out, where=den != 0)
    return out


def curve_metrics(cm, thresholds) -> dict:
    """PR curve, ROC, AP and AUROC of ``cm [T, 2, 2]`` at ``thresholds [T]``, in float64:

    * ``pr_curve`` = (precision, recall, thresholds): precision = tp / (tp + fp), 1.0 on 0 / 0 (current torchmetrics'
      zero_division; older versions gave 0); recall = tp / (tp + fn), 0 on 0 / 0; then precision 1 and recall 0 appended;
    * ``ap`` = -sum_k (recall[k+1] - recall[k]) * precision[k] over those T + 1 points;
    * ``roc`` = (fpr, tpr, thresholds), each flipped: tpr = tp / (tp + fn), fpr = fp / (fp + tn), 0 on 0 / 0;
    * ``auroc`` = trapz(tpr, fpr) over those T points, no end points added (torchmetrics' _auc_compute_without_check)."""
    cm = np.asarray(cm, np.int64)
    thr = np.asarray(thresholds, np.float32)
    tp, fp, fn, tn = cm[:, 1, 1], cm[:, 0, 1], cm[:, 1, 0], cm[:, 0, 0]
    precision = np.concatenate([_div(tp, tp + fp, 1.0), [1.0]])
    recall = np.concatenate([_div(tp, tp + fn, 0.0), [0.0]])
    ap = float(-np.sum((recall[1:] - recall[:-1]) * precision[:-1]))
    tpr = _div(tp, tp + fn, 0.0)[::-1].copy()
    fpr = _div(fp, fp + tn, 0.0)[::-1].copy()
    auroc = float(np.sum((fpr[1:] - fpr[:-1]) * (tpr[1:] + tpr[:-1]) / 2.0))
    return {"pr_curve": (precision, recall, thr.copy()), "roc": (fpr, tpr, thr[::-1].copy()), "ap": ap, "auroc": auroc}
