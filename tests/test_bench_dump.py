"""`bench.py --dump-outputs`: the files it writes (CPU), and on the GPU that they are the outputs of the last timed step,
with the shared counters summed over exactly `--steps` steps (against the oracle)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import bench
from btpost import synth
from oracle import oracle

ROOT = Path(__file__).resolve().parents[1]


def _outputs():
    return {"det_count": torch.tensor([3, 0], dtype=torch.int32), "det_keep": torch.tensor([[7, -1], [2**40, 5]]),
            "dets": torch.linspace(-1, 1, 12).reshape(2, 1, 6), "mask": torch.arange(64, dtype=torch.uint8).reshape(8, 8),
            "sum": torch.tensor([0.1, 1e300], dtype=torch.float64), "big": torch.arange(5000, dtype=torch.int32),
            "bits": torch.arange(3000, dtype=torch.int64).reshape(30, 100) % 256}


def _load(d):
    return {p.stem: np.load(p) for p in sorted(Path(d).glob("*.npy"))}


def test_dump_keeps_every_value_and_shape(tmp_path):
    out = _outputs()
    assert bench.dump_outputs(out, tmp_path / "a") == []
    got = _load(tmp_path / "a")
    assert set(got) == set(out)
    for k, t in out.items():
        wide = t.dtype in (torch.int32, torch.int64, torch.float64)
        assert got[k].dtype == (np.float64 if wide else np.float32), k
        assert got[k].shape == tuple(t.shape), k
        np.testing.assert_array_equal(got[k], t.numpy().astype(got[k].dtype))
        assert (got[k] == t.numpy()).all(), k                    # the conversion lost nothing


def test_dump_over_budget_samples_the_largest_outputs(tmp_path):
    out, budget = _outputs(), 40_000
    cut = bench.dump_outputs(out, tmp_path / "a", budget=budget)
    assert cut == ["big", "bits"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").glob("*.npy")) <= budget
    got = _load(tmp_path / "a")
    for k in ("det_count", "det_keep", "dets", "mask", "sum"):   # the small outputs stay whole
        np.testing.assert_array_equal(got[k], out[k].numpy())
    idx = got["big"]                                             # value == flat index: the sample is distinct, ascending
    assert idx.ndim == 1 and 0 < len(idx) < 5000 and (np.diff(idx) > 0).all() and idx[-1] < 5000
    assert got["bits"].ndim == 1 and 0 < len(got["bits"]) < 3000
    bench.dump_outputs(out, tmp_path / "b", budget=budget)       # same arguments, same sample
    for k, v in _load(tmp_path / "b").items():
        assert v.tobytes() == got[k].tobytes(), k


@pytest.mark.gpu
def test_dump_is_the_last_timed_step(tmp_path):
    B, S, steps = 4, 160, 7
    cmd = [sys.executable, str(ROOT / "bench.py"), "--steps", str(steps), "--warmup", "2", "--batch", str(B), "--img", str(S),
           "--no-e2e", "--cpu-sample", "0", "--clock-period-ms", "0", "--dump-outputs", str(tmp_path)]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    depth, warmup = line["config"]["batches_in_flight"], line["warmup"]
    slots = [(warmup + i) % depth for i in range(steps)]         # round robin, continuing after the warm-up steps
    refs = {s: oracle.run_pipeline(synth.make_batch(synth.SynthConfig(batch=B, img_size=S, seed=bench.SEED, image_offset=s * B)),
                                   img_size=S) for s in set(slots)}
    got, ref = _load(tmp_path), refs[slots[-1]]
    for k in ("n_cand", "det_count", "det_keep", "det_anchor", "dets", "det_coeff", "gt_count", "gt_boxes", "gt_boxes_raw",
              "gt_labels", "cm_pos", "seg_img3", "uni_img3", "inst_area", "inst_inter", "dt_match", "dt_ignore", "gt_ignore"):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
    for k in ("seg_dice", "seg_iou", "uni_dice", "uni_iou"):
        np.testing.assert_allclose(got[k], ref[k], rtol=1e-5, err_msg=k)
    for k in ("cm", "seg_cnt4", "uni_cnt4"):                     # shared by the slots: one term per timed step
        np.testing.assert_array_equal(got[k], sum(refs[s][k] for s in slots), err_msg=k)
