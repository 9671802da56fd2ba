"""CPU: the oracle against the float64 restatement of tests/f64_reference.py at image sizes and class counts the
CUDA tests reach only through the oracle -- a prototype width below one 32-column tile (S = 32, 96), partial tiles of
16 and 24 columns (S = 320, 480), one class and sixteen.  The oracle is pinned against torch elsewhere only at 160^2
and 640^2 with three classes."""
import numpy as np
import pytest

import f64_reference as f64
import helpers
from oracle import oracle

SIZES = (32, 96, 320, 480)
CLASSES = (1, 3, 16)


@pytest.mark.parametrize("nc", CLASSES)
@pytest.mark.parametrize("S", SIZES)
def test_oracle_matches_float64_reference(S, nc):
    batch = helpers.make(batch=2, img_size=S, seed=20286, nc=nc)
    max_det = 300 if S <= 320 else 100
    ref = helpers.oracle_parallel(batch, img_size=S, nc=nc, max_det=max_det)
    assert int(ref["det_count"].min()) > 0 and int(ref["gt_count"].min()) > 0 and int(batch["masks_gt"].sum()) > 0
    labels = f64.check_l2_detections(batch["head"], ref, nc, S)
    if nc == 16:
        assert labels.max() >= 8
    _, _, n_band = f64.check_projector(batch["protos"], batch["proj_weight"], batch["proj_bias"], batch["masks_gt"], ref, S)
    assert n_band <= 1e-3 * 2 * S * S, n_band
    n_inst = f64.check_instances(batch["protos"], ref, lambda b: ref["inst_masks"][b], S)
    assert n_inst <= 1e-3 * int(ref["det_count"].sum()) * S * S, n_inst


def test_float64_reference_catches_a_wrong_crop_column():
    """The instance check is not vacuous: one more prototype column kept at the right edge of a crop box (what a
    16- or 24-column tile edge handled wrongly would produce) is reported."""
    S = 96
    batch = helpers.make(batch=1, img_size=S, seed=20281)
    ref = oracle.run_pipeline(batch, img_size=S, max_det=20)
    wide = dict(ref, dets=ref["dets"].copy())
    wide["dets"][0, :, 2] += 4.0                      # x2 one prototype pixel further right
    bad = [oracle.instance_mask(batch["protos"][0], ref["det_coeff"][0, i], wide["dets"][0, i, :4], S)
           for i in range(int(ref["det_count"][0]))]
    with pytest.raises(AssertionError, match="instance masks"):
        f64.check_instances(batch["protos"], ref, lambda b: np.stack(bad), S)
