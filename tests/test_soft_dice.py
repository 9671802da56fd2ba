"""CPU: v3's soft Dice on the projector probabilities (BtIOSoftDice.seg_soft2 / seg_soft_dice / seg_soft_acc) -- the ABI
layout of the new fields, their argument validation (before any CUDA call), the numpy restatement's exp against the oracle's C
exp, and the restatement against the reference's own formula (SURVEY.md A.4 with torch.sigmoid) on the reference's
upsampled logits."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

import soft_dice_oracle as sd
from btpost import _lib, synth
from oracle import oracle

ROOT = Path(__file__).resolve().parents[1]
GOLD = ROOT / "tests" / "golden"


def test_soft_dice_io_layout(tmp_path):
    """BtIO keeps its layout; BtIOSoftDice is a BtIO followed by the three outputs, selected by BtParams.io_soft_dice,
    which takes one of BtParams' reserved words (same size, every other offset unchanged)."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "btpost.h"\nint main(){'
                   'printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(BtIO), sizeof(BtIOSoftDice), offsetof(BtIOSoftDice, io), '
                   'offsetof(BtIOSoftDice, seg_soft2), offsetof(BtIOSoftDice, seg_soft_dice), offsetof(BtIOSoftDice, seg_soft_acc), '
                   'sizeof(BtParams), offsetof(BtParams, io_soft_dice));return 0;}')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    S = _lib.BtIOSoftDice
    assert got == [C.sizeof(_lib.BtIO), C.sizeof(S), 0, S.seg_soft2.offset, S.seg_soft_dice.offset, S.seg_soft_acc.offset,
                   C.sizeof(_lib.BtParams), _lib.BtParams.io_soft_dice.offset]
    assert _lib._IO_FIELDS[-1] == "seg_sweep" and got[0] == 8 * len(_lib._IO_FIELDS)
    assert got[3:6] == [got[0], got[0] + 8, got[0] + 16] and got[1] == got[0] + 24
    assert got[7] == _lib.BtParams.in_flight.offset + 4 and got[6] == got[7] + 8 == _lib.BtParams.reserved.offset + 4


def _params():
    p = _lib.BtParams()
    p.batch, p.num_anchors, p.nc, p.nm, p.max_det, p.max_gt = 2, 8400, 3, 32, 300, 32
    p.img_h = p.img_w = 640
    p.proto_h = p.proto_w = 160
    p.num_iou_thrs = 10
    n = C.c_size_t()
    assert _lib.load().btpost_workspace_bytes(C.byref(p), C.byref(n)) == 0
    return p, n.value


def test_soft_dice_argument_validation_without_gpu():
    """seg_soft_dice and seg_soft_acc are computed from seg_soft2: either one without it is BT_ERR_BAD_ARG, and so is an
    io_soft_dice other than 0 / 1; all are returned by the mask stage and by btpost_run before any CUDA call."""
    L = _lib.load()
    p, ws = _params()
    io = _lib.BtIOSoftDice()
    for f in ("head", "protos", "masks_gt", "proj_weight", "dets", "det_count", "det_coeff", "det_keep", "det_anchor", "n_cand",
              "gt_count", "gt_boxes", "gt_boxes_raw", "gt_labels", "cm", "cm_pos"):
        setattr(io, f, 4096)
    masks = lambda: L.btpost_masks_parts(C.byref(p), C.byref(io), C.c_void_p(256), ws, None, _lib.MASKS_CELLS)
    run = lambda: L.btpost_run(C.byref(p), C.byref(io), C.c_void_p(256), ws, None)
    p.io_soft_dice = 1
    io.seg_soft_dice = 4096                                          # seg_soft2 missing
    assert masks() == -1 and run() == -1
    io.seg_soft_dice, io.seg_soft_acc = None, 4096                   # seg_soft2 missing
    assert masks() == -1 and run() == -1
    io.seg_soft_dice = 8192
    assert masks() == -1 and run() == -1
    p.io_soft_dice = 2                                               # neither a BtIO nor a BtIOSoftDice
    io.seg_soft2 = 4096
    assert masks() == -1 and run() == -1


def test_numpy_exp_is_the_oracle_exp():
    """The restatement's fma-only exp equals oracle/btpost_oracle.c::bto_expf bit for bit over the range the sigmoid
    uses (and returns 0 below -87 like it)."""
    rng = np.random.default_rng(7)
    xs = np.concatenate([np.linspace(-90.0, 87.0, 40001, dtype=np.float32), rng.uniform(-87.0, 87.0, 20000).astype(np.float32),
                         rng.normal(0.0, 2.0, 20000).astype(np.float32),
                         np.array([-87.0, np.nextafter(np.float32(-87.0), np.float32(0.0)), -86.99, 0.0, -0.0, 1e-30, -1e-30,
                                   0.5, -0.5, 87.0], np.float32)])
    got = sd.bt_expf(xs)
    f = oracle.lib().bto_expf_public
    want = np.array([f(float(x)) for x in xs], np.float32)
    assert got.tobytes() == want.tobytes()


def test_soft_prob_edges():
    x = np.array([-1000.0, -87.5, np.nextafter(np.float32(-87.0), np.float32(-100.0)), -87.0, 0.0, 87.0, 88.0, 1000.0], np.float32)
    p = sd.soft_prob(x)
    assert (p[:3] == 0).all() and 0 < p[3] < 2.0 ** -125 and p[4] == 0.5 and (p[5:] == 1.0).all()
    q = np.rint(p.astype(np.float64) * sd.FX)
    assert q[3] == 0 and q[4] == 2.0 ** 39 and q[-1] == 2.0 ** 40


@pytest.mark.parametrize("name", ["ref_v3_s160", "ref_v3_s160_loose", "ref_v3_s160_peaked"])
def test_oracle_soft_dice_follows_the_reference_formula(name):
    """On the reference's own upsampled logits: per image 2 sum(p t) / (sum p + sum t) with p = torch.sigmoid -- what
    the reference passes to DiceScore -- agrees with the restatement within 1e-6 relative."""
    f = np.load(GOLD / f"{name}.npz")
    cfg = synth.SynthConfig(batch=int(f["batch"]), img_size=int(f["img_size"]), seed=int(f["seed"]))
    batch = synth.make_batch(cfg, l1=True, l1_peaked=bool(int(f["l1_peaked"])))
    logits, gt = f["seg_logits"], batch["masks_gt"][:, 0] != 0
    soft2 = sd.soft_sums(logits, gt)
    got = sd.soft_dice(soft2, gt.reshape(len(gt), -1).sum(1))
    p = torch.from_numpy(logits).sigmoid().double().numpy()
    t = gt.astype(np.float64)
    want = 2 * (p * t).sum((1, 2)) / (p.sum((1, 2)) + t.sum((1, 2)))
    assert np.isfinite(got).all() and (want > 0).all()
    np.testing.assert_allclose(got, want, rtol=1e-6)
    np.testing.assert_allclose(soft2[:, 1] / sd.FX, p.sum((1, 2)), rtol=1e-6)
