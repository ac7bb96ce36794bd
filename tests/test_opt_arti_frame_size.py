"""``tools.opt_arti`` takes the camera from the records' frame size and refuses a file that mixes sizes before
any device work (CPU only)."""
import os

import pytest
import torch

from articulation3d_b200 import adapter, io, opt_utils
from articulation3d_b200.tools import opt_arti


def _records(video_id, size, frames=3):
    h, w = size
    return [{"image_id": t, "file_name": f"{video_id}_{t}.png",
             "instances": [{"image_id": t, "category_id": 0, "bbox": [1.0, 1.0, 4.0, 4.0], "score": 0.9,
                            "segmentation": {"size": [h, w], "counts": f"{h * w}"}}],
             "pred_plane": torch.zeros(1, 3), "pred_rot_axis": torch.zeros(1, 3), "pred_tran_axis": torch.zeros(1, 2)}
            for t in range(frames)]


def test_frame_config_follows_segmentation_size():
    cfg = opt_arti.frame_config(adapter.group_by_video(_records("synthetic00_0_0", (480, 640))))
    assert (cfg.height, cfg.width, cfg.focal_length) == (480, 640, 517.97)
    cfg = opt_arti.frame_config(adapter.group_by_video(_records("synthetic00_0_0", (768, 1024))))
    assert (cfg.height, cfg.width, cfg.focal_length) == (768, 1024, 517.97 * 1024 / 640)
    empty = _records("synthetic00_0_0", (768, 1024))
    for r in empty:
        r["instances"] = []
    assert opt_arti.frame_config(adapter.group_by_video(empty)).width == 640


def test_mixed_frame_sizes_refused_before_device_work(tmp_path, monkeypatch):
    path, out = str(tmp_path / "mixed.pth"), str(tmp_path / "out")
    torch.save(_records("synthetic00_0_0", (480, 640)) + _records("synthetic01_0_0", (768, 1024)), path)

    def no_device_work(*a, **k):
        raise AssertionError("reached the optimisation")
    for mod, name in ((io, "records_to_preds"), (opt_utils, "track_planes"), (opt_utils, "optimize_videos")):
        monkeypatch.setattr(mod, name, no_device_work)
    monkeypatch.delenv("WORLD_SIZE", raising=False)
    with pytest.raises(ValueError) as e:
        opt_arti.main(["--input", path, "--output", out])
    msg = str(e.value)
    assert "[480, 640]" in msg and "synthetic00_0_0" in msg and "[768, 1024]" in msg and "synthetic01_0_0" in msg
    assert not os.path.exists(out)


def test_legacy_format_loads_with_mmap(tmp_path):
    """torch's legacy (non-zip) format cannot be memory-mapped: the loader under torchrun reads it instead."""
    recs = _records("synthetic00_0_0", (480, 640))
    path = str(tmp_path / "legacy.pth")
    torch.save(recs, path, _use_new_zipfile_serialization=False)
    got = adapter.load_predictions(path, mmap=True)
    assert [r["file_name"] for r in got] == [r["file_name"] for r in recs]
    assert torch.equal(got[0]["pred_plane"], recs[0]["pred_plane"])
