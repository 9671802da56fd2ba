"""TEST INFRASTRUCTURE ONLY -- numpy restatement of btpost_seg_curve (the binned PR / ROC state of the projector
probabilities, DESIGN.md §4): from the upsampled projector logits, the GT masks and the fp32 thresholds, hist [2, T+1]
int64 with hist[t][j] = pixels with GT value t (gt != 0) and exactly j thresholds <= p, p = soft_dice_oracle.soft_prob
(the kernel's sigmoid, pinned in tests/test_soft_dice.py).  A NaN p is below every threshold."""
import numpy as np

from soft_dice_oracle import soft_prob


def bins(p, thresholds):
    """Number of thresholds <= p for each p (thresholds non-decreasing; NaN p -> 0)."""
    thr = np.asarray(thresholds, np.float32)
    p = np.asarray(p, np.float32).reshape(-1)
    j = np.searchsorted(thr, p, side="right")
    return np.where(np.isnan(p), 0, j)


def hist_from_probs(p, gt, thresholds):
    t = (np.asarray(gt) != 0).reshape(-1).astype(np.int64)
    T = len(thresholds)
    key = t * (T + 1) + bins(p, thresholds)
    return np.bincount(key, minlength=2 * (T + 1)).reshape(2, T + 1).astype(np.int64)


def seg_curve_hist(logits, gt, thresholds):
    """[B, S, S] upsampled logits, [B, S, S] (or [B, 1, S, S]) GT -> hist [2, T+1] int64."""
    return hist_from_probs(soft_prob(logits), gt, thresholds)
