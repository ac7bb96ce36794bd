"""``adapter.override_depth_records`` and ``tools.opt_arti --override-depth`` refuse records they cannot override
before any library load or device use; synthetic depth (``synth.render_depths``) and its records (CPU only)."""
import os

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, adapter, engine, io, opt_utils, rle, synth
from articulation3d_b200.tools import opt_arti
from oracle import restated


def _records(video_id="synthetic00_0_0", size=(48, 64), frames=3, n=2):
    h, w = size
    return [{"image_id": t, "file_name": f"{video_id}_{t}.png",
             "instances": [{"image_id": t, "category_id": 0, "bbox": [1.0, 1.0, 4.0, 4.0], "score": 0.9,
                            "segmentation": {"size": [h, w], "counts": f"{h * w}"}} for _ in range(n)],
             "pred_plane": torch.ones(n, 3), "pred_rot_axis": torch.zeros(n, 3), "pred_tran_axis": torch.zeros(n, 2),
             "pred_depth": torch.ones(h, w)}
            for t in range(frames)]


def _no_device(monkeypatch):
    def fail(*a, **k):
        raise AssertionError("reached the library or the device")
    for mod, name in ((_lib, "load"), (engine, "rle_to_pool"), (engine, "plane_offsets"),
                      (io, "records_to_preds"), (opt_utils, "track_planes"), (opt_utils, "optimize_videos")):
        monkeypatch.setattr(mod, name, fail)


def _broken(kind):
    recs = _records()
    bad = recs[1]
    if kind == "no_depth":
        del bad["pred_depth"]
    elif kind == "depth_shape":
        bad["pred_depth"] = torch.ones(64, 48)
    elif kind == "plane_rows":
        bad["pred_plane"] = torch.ones(3, 3)
    return recs, bad["file_name"]


KINDS = pytest.mark.parametrize("kind,words", [("no_depth", "pred_depth"), ("depth_shape", "[64, 48]"),
                                                ("plane_rows", "pred_plane")])


@KINDS
def test_function_refuses_before_device_work(kind, words, monkeypatch):
    recs, name = _broken(kind)
    _no_device(monkeypatch)
    planes = [r["pred_plane"].clone() for r in recs]
    with pytest.raises(ValueError) as e:
        adapter.override_depth_records(recs, "cuda:0")
    assert name in str(e.value) and words in str(e.value)
    assert all(torch.equal(r["pred_plane"], p) for r, p in zip(recs, planes))        # nothing swapped yet


@KINDS
def test_tool_refuses_before_device_work(kind, words, tmp_path, monkeypatch):
    recs, name = _broken(kind)
    recs += _records("synthetic01_0_0")
    path, out = str(tmp_path / "pred.pth"), str(tmp_path / "out")
    torch.save(recs, path)
    _no_device(monkeypatch)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    with pytest.raises(ValueError) as e:
        opt_arti.main(["--input", path, "--output", out, "--override-depth"])
    assert name in str(e.value) and words in str(e.value)
    assert not os.path.exists(out)


def test_records_without_instances_need_no_size_match():
    recs = _records(n=0)
    recs[0]["pred_depth"] = torch.ones(3, 5)
    adapter.check_depth_records(recs)
    with pytest.raises(ValueError, match="mix frame sizes"):
        r = _records(n=2)
        r[0]["instances"][1]["segmentation"] = {"size": [49, 64], "counts": f"{49 * 64}"}
        adapter.check_depth_records(r)


def test_synthetic_depth_is_deterministic_finite_positive_with_background():
    preds, scene = synth.make_video(31, 3, 5)
    d = synth.render_depths(scene, background=7.5)
    _, scene2 = synth.make_video(31, 3, 5)
    assert d.shape == (5, 480, 640) and d.dtype == torch.float32
    assert torch.equal(d, synth.render_depths(scene2, background=7.5))
    assert torch.isfinite(d).all() and (d > 0).all()
    cfg = OptConfig()
    covered = torch.stack([synth.render_track_masks(scene, k, cfg) for k in range(3)]).any(0)
    assert covered.any() and (~covered).any()
    assert (d[~covered] == 7.5).all() and (d[covered] < 7.5).all()
    assert not torch.equal(d, synth.render_depths(synth.make_video(32, 3, 5)[1], background=7.5))


def test_synthetic_depth_gives_back_the_true_planes_on_the_oracle():
    """The reference's ``override_depth`` (CPU restatement) of records holding the scene's true planes returns
    them: every mask pixel's depth lies on its own plane."""
    preds, scene = synth.make_video(2020, 4, 6)
    d = synth.render_depths(scene)
    true = synth.scene_pred_planes(scene)
    rays = torch.FloatTensor(adapter.get_K_inv_dot_xy_1())
    for t, p in enumerate(preds):
        inst = {"instances": [{"segmentation": rle.encode(m.numpy() > 0.5)} for m in p.pred_masks],
                "pred_plane": true[:, t].clone()}
        got = restated.override_depth(rays * d[t], inst)["pred_plane"]
        np.testing.assert_allclose(got.numpy(), true[:, t].numpy(), rtol=1e-4, atol=1e-6)


def test_preds_to_records_stores_depth():
    preds, scene = synth.make_video(5, 2, 3)
    d = synth.render_depths(scene)
    recs = io.preds_to_records(preds, depths=d)
    assert all(torch.equal(r["pred_depth"], d[t]) and r["pred_depth"].dtype == torch.float32
               for t, r in enumerate(recs))
    assert "pred_depth" not in io.preds_to_records(preds)[0]
    # the optimised records carry the input's depth on
    assert torch.equal(io.opt_preds_to_records(io.records_to_preds(recs[:1]), recs[:1])[0]["pred_depth"], d[0])


def test_synthetic_depth_needs_synthetic(tmp_path):
    with pytest.raises(SystemExit):
        opt_arti.main(["--input", str(tmp_path / "x.pth"), "--output", str(tmp_path / "o"), "--synthetic-depth"])
