"""Pins the CPU oracle (oracle/restated.py) against the committed fixtures in
tests/golden/ — outputs of the UNMODIFIED reference run under oracle/ref_shim.py
(oracle/gen_golden.py regenerates them where the reference sources exist).
"""
import random

import numpy as np
import pytest
import torch

from articulation3d_b200.structures import Boxes, Instances
from oracle import restated
from tests import golden_util as gu


class _Rec:
    def __init__(self):
        self.choices = []

    def choice(self, seq):
        c = random.choice(seq)
        self.choices.append((int(c), len(seq)))
        return c


def run_restated(preds, seed, monkeypatch):
    rec, lin = _Rec(), []
    real = restated.linregress

    def linregress(x, y):
        lin.append(np.asarray(y, dtype=np.float32).copy())
        return real(x, y)

    monkeypatch.setattr(restated, "random", rec)
    monkeypatch.setattr(restated, "linregress", linregress)
    random.seed(seed)
    planes = restated.track_planes(preds)
    trace = []
    out = restated.optimize_planes(preds, planes, "3dc", trace=trace)
    return planes, out, rec.choices, lin, trace


@pytest.mark.parametrize("name", gu.golden_cases())
def test_restated_oracle_matches_golden(name, monkeypatch):
    z = gu.load(name)
    preds = gu.arrays_to_preds(z, Instances, Boxes)
    planes, out, choices, lin, trace = run_restated(preds, int(z["seed"]), monkeypatch)
    gu.check_against_golden(z, planes, out, choices, lin)
    # the quantities the reference never exposes must be self-consistent
    for step in trace:
        for v in step["visits"]:
            iou = v["inter"].astype(np.float32) / v["union"].astype(np.float32)
            assert np.array_equal(iou, v["iou"], equal_nan=True)


def test_golden_covers_both_outcomes():
    seen = set()
    for name in gu.golden_cases():
        z = gu.load(name)
        for cat in ("trans", "rot"):
            for i in range(int(z[f"{cat}_n"])):
                seen.add((cat, bool(z[f"{cat}{i}_has_rot"])))
    assert ("rot", True) in seen and ("rot", False) in seen and ("trans", True) in seen


@pytest.mark.parametrize("name", ["depth_a", "depth_b"])
def test_override_depth_oracle_matches_reference_fixture(name, golden_dir):
    """Row f1: oracle/restated.override_depth / get_K_inv_dot_xy_1 against the outputs of the reference's own
    static ``PlaneRCNN_Branch.override_depth`` (utils/arti_vis.py:101-149), tests/golden/depth/*.npz."""
    import os
    import torch
    from oracle import restated
    from oracle.gen_golden import depth_case_inputs
    z = np.load(os.path.join(golden_dir, "depth", f"{name}.npz"))
    records, depths = depth_case_inputs(name)
    assert float(depths.astype(np.float64).sum()) == float(z["depth_checksum"])      # same inputs as the generator's
    rays64 = restated.get_K_inv_dot_xy_1()
    assert np.array_equal(rays64[:, ::37, ::41], z["rays_probe"])
    rays = torch.FloatTensor(rays64)
    assert len(records) == int(z["n_frames"])
    for i, rec in enumerate(records):
        assert np.array_equal(rec["pred_plane"].numpy(), z[f"f{i}_pred_plane_in"])
        out = restated.override_depth(rays * torch.from_numpy(depths[i]),
                                      {"instances": rec["instances"], "pred_plane": rec["pred_plane"].clone()})
        np.testing.assert_allclose(out["pred_plane"].numpy(), z[f"f{i}_pred_plane_out"], rtol=1e-6, atol=1e-7)
