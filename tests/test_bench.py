"""bench.py --dump-outputs: what the timed steps computed, written so that two builds can be compared output for
output, and --steps as the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from tests import golden_util as gu


def test_dump_arrays_keeps_the_budget_and_the_values():
    big = torch.arange(3000 * 480 * 20, dtype=torch.int32).reshape(3000, 480, 20)
    arrays = {"ints": torch.tensor([1, -2, 2 ** 31 - 1], dtype=torch.int32), "f32": torch.rand(1000),
              "f64": torch.rand(10, dtype=torch.float64), "big": big, "empty": torch.zeros(0, 3)}
    budget = 8 * 10 ** 6
    got = bench.dump_arrays(arrays, budget)
    assert sum(a.nbytes + bench.NPY_HEADER for a in got.values()) <= budget
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["ints"].tolist() == [1, -2, 2 ** 31 - 1]
    assert np.array_equal(got["f32"], arrays["f32"].numpy()) and np.array_equal(got["f64"], arrays["f64"].numpy())
    assert got["empty"].shape == (0, 3)
    rows = got["big_rows"].astype(np.int64)
    assert 0 < len(rows) < 3000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(got["big"], big.numpy()[rows].astype(np.float64))
    again = bench.dump_arrays(arrays, budget)
    assert sorted(again) == sorted(got) and all(np.array_equal(again[k], got[k]) for k in got)


def _run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(gu.ROOT, "bench.py"), "--workload", "c2", "--steps", str(steps),
           "--warmup", "1", "--e2e-videos", "1", "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(out_dir)]
    proc = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-4000:]
    line = json.loads([ln for ln in proc.stdout.splitlines() if ln.startswith("{")][-1])
    files = sorted(os.listdir(out_dir))
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}, \
        sum(os.path.getsize(os.path.join(out_dir, f)) for f in files)


@pytest.mark.gpu
def test_bench_dumps_the_same_outputs_every_run(tmp_path):
    line, a, nbytes = _run_bench(tmp_path / "a", 3)
    assert line["steps"] == 3 and len(line["e2e"]["ms_each_step"]) == 3
    assert nbytes <= bench.DUMP_BYTES
    for name in ("best_cand", "best_inter", "best_union", "best_iou", "proj_bits", "proj_popc", "proj_bbox"):
        assert "pass_" + name in a
    for name in ("scores", "pred_planes", "pred_rot_axis", "pred_tran_axis", "frame_records", "track_records"):
        assert "e2e_" + name in a
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert len(a["pass_best_cand"]) == line["config"]["units_per_step"] // 90        # one per track-frame
    assert len(a["e2e_frame_records"]) > 0
    line_b, b, _ = _run_bench(tmp_path / "b", 2)
    assert line_b["steps"] == 2 and len(line_b["e2e"]["ms_each_step"]) == 2
    assert sorted(a) == sorted(b)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
