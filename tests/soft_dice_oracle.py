"""TEST INFRASTRUCTURE ONLY -- numpy restatement of v3's soft Dice on the projector probabilities (SURVEY.md A.4,
`/root/reference/src/running_main_v3.py:466-474`) with the CUDA library's arithmetic, so that tests can compare
`seg_soft2` bit for bit and `seg_soft_dice` / the accumulator exactly:

- p = 1 / (1 + exp(-x)) in fp32 with the oracle's fma-only exp (`oracle/btpost_oracle.c::bto_expf`, pinned against
  it in tests/test_soft_dice.py) and one rounding per operation; p = 0 for x < -87;
- each p rounded to 2^-40 fixed point (int64), summed over the S^2 pixels (sum p) and over the GT pixels (sum p * t);
- soft Dice = 2 A / (P + G) in double, rounded to fp32, NaN when P + G == 0; the accumulator adds
  round(soft Dice * 2^40) and counts the images with a defined value."""
import numpy as np

FX = float(2 ** 40)


def fma32(a, b, c):
    """fp32 fmaf(a, b, c), correctly rounded.  The product of two fp32 values is exact in float64; the sum is rounded
    to odd in float64 (TwoSum gives the exact remainder), and 53 >= 24 + 2 bits make the final rounding to fp32 the
    single rounding of the fused operation."""
    a, b, c = (np.asarray(v, np.float32).astype(np.float64) for v in (a, b, c))
    p = a * b
    s = p + c
    bv = s - p
    err = (p - (s - bv)) + (c - bv)
    even = (s.view(np.int64) & 1) == 0
    s = np.where((err != 0) & even, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def bt_expf(x):
    """oracle/btpost_oracle.c::bto_expf elementwise (Cody-Waite reduction + degree-6 polynomial)."""
    x = np.asarray(x, np.float32)
    t = x * np.float32(1.4426950408889634)
    n = np.rint(t)
    r = fma32(n, np.float32(-0.693145751953125), x)
    r = fma32(n, np.float32(-1.428606765330187e-06), r)
    p = np.full_like(x, np.float32(1.3888889225e-03))
    for c in (8.3333337680e-03, 4.1666667908e-02, 1.6666667163e-01, 0.5, 1.0, 1.0):
        p = fma32(p, r, np.float32(c))
    with np.errstate(invalid="ignore"):
        e = np.where(x < np.float32(-87.0), 0, n).astype(np.int32)
    out = (p.view(np.int32) + (e << 23)).view(np.float32)
    return np.where(x < np.float32(-87.0), np.float32(0.0), out)


def soft_prob(x):
    """sigmoid(x) in fp32 as the kernel computes it; 0 for x < -87."""
    x = np.asarray(x, np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        p = np.float32(1.0) / (np.float32(1.0) + bt_expf(np.where(x < np.float32(-87.0), np.float32(0.0), -x)))
    return np.where(x < np.float32(-87.0), np.float32(0.0), p).astype(np.float32)


def soft_sums(logits, gt):
    """[B, S, S] upsampled projector logits and GT masks -> [B, 2] int64 (sum p * t, sum p) in units of 2^-40."""
    q = np.rint(soft_prob(logits).astype(np.float64) * FX).astype(np.int64)
    t = np.asarray(gt) != 0
    B = q.shape[0]
    return np.stack([np.where(t, q, 0).reshape(B, -1).sum(1), q.reshape(B, -1).sum(1)], 1)


def soft_dice(soft2, n_gt):
    """[B, 2] fixed-point sums and [B] |G| -> [B] fp32 soft Dice (NaN when P + G == 0)."""
    a, p = soft2[:, 0].astype(np.float64), soft2[:, 1].astype(np.float64)
    g = np.asarray(n_gt, np.int64)
    defined = (soft2[:, 1] != 0) | (g != 0)
    with np.errstate(invalid="ignore", divide="ignore"):
        d = (2.0 * a / (p + g.astype(np.float64) * FX)).astype(np.float32)
    return np.where(defined, d, np.float32(np.nan))


def accumulate(dice):
    """What the kernel adds to seg_soft_acc for the images of `dice`: (sum of round(d * 2^40), count)."""
    d = np.asarray(dice, np.float32)
    ok = ~np.isnan(d)
    return np.array([int(np.rint(d[ok].astype(np.float64) * FX).astype(np.int64).sum()), int(ok.sum())], np.int64)


def mean(acc):
    """DeviceSweep.finish()'s seg_soft_dice from an accumulator (sum, count)."""
    s, k = int(acc[0]), int(acc[1])
    return s / FX / k if k else float("nan")
