"""CPU restatement of btpost_surface_distance (include/btpost.h, DESIGN.md §4): MONAI's compute_hausdorff_distance and
compute_average_surface_distance (symmetric=True) with their version-dependent choices fixed, on scipy.ndimage and
torch.quantile.  Per image, P = pred != 0 and G = gt != 0:

  edges      edge(M) = M AND NOT binary_erosion(M) (scipy's defaults: 4-neighbour cross, background outside the image),
             as MONAI's get_mask_edges applies it (its crop to the union's bounding box changes no distance)
  distances  distance_transform_edt(~edge(G))[edge(P)] and the same from G to P
  hd         the largest distance of either direction
  hd95       max of torch.quantile(d.double(), 0.95) over the two directions
  assd       mean of both directions' distances together
  undefined  P or G empty: NaN in all three (MONAI returns inf or nan there, depending on its version), not counted

The library rounds each value once to fp32; the accumulator words are sums of round(value * 2^32) over the images with
defined values, and their count."""
import numpy as np
import torch
from scipy import ndimage

ACC = 2.0 ** 32


def edges(mask):
    m = np.asarray(mask) != 0
    return m & ~ndimage.binary_erosion(m)


def directed(a_edges, b_edges):
    """Distance from every edge pixel of a to the nearest edge pixel of b (float64, in the row-major order of a's edges)."""
    return ndimage.distance_transform_edt(~b_edges)[a_edges]


def q95(d):
    return float(torch.quantile(torch.from_numpy(np.asarray(d, np.float64)), 0.95))


def surface_distance(pred, gt):
    """(hd, hd95, assd) in float64 for one S x S pair; NaN for all three when either mask is empty."""
    ep, eg = edges(pred), edges(gt)
    if not ep.any() or not eg.any():
        return float("nan"), float("nan"), float("nan")
    dp, dg = directed(ep, eg), directed(eg, ep)
    return max(dp.max(), dg.max()), max(q95(dp), q95(dg)), float(np.concatenate([dp, dg]).mean())


def surface_batch(pred, gt):
    """pred [B, S, S], gt [B, S, S] or [B, 1, S, S] -> (hd, hd95, assd) fp32 [B], as the library returns them."""
    gt = np.asarray(gt).reshape(np.asarray(pred).shape)
    vals = np.array([surface_distance(p, g) for p, g in zip(pred, gt)], np.float64).reshape(-1, 3)
    return tuple(vals[:, i].astype(np.float32) for i in range(3))


def accumulate(hd, hd95, assd):
    """The accumulator words [4] of a set of per-image fp32 values: sums of round(v * 2^32), count of defined images."""
    ok = ~np.isnan(hd)
    words = [int(np.rint(np.asarray(v, np.float64)[ok] * ACC).astype(np.int64).sum()) for v in (hd, hd95, assd)]
    return np.array(words + [int(ok.sum())], np.int64)


def means(acc):
    """(hd, hd95, assd) means from the accumulator words, NaN when no image had defined values (DeviceSweep.finish)."""
    n = int(acc[3])
    return tuple(int(acc[i]) / ACC / n if n else float("nan") for i in range(3))
