"""``tools.opt_arti`` over the GPUs of one box under torchrun, against a one-GPU run of the same input: the same
files with equal contents, the same AP lines printed once, the summary's evaluation count; a rank with no video;
``--device`` refused under torchrun.  Records at 1024x768 get the camera of their frame size.

Every torchrun case runs twice: ``nccl``, the tool as users launch it, one rank per GPU (needs 2 GPUs); and
``one_gpu``, both ranks on cuda:0 over gloo (``tests/one_gpu_ranks.py``), so the distributed path runs on a box
with a single GPU too."""
import json
import os
import re
import signal
import subprocess
import sys
from contextlib import redirect_stdout
from io import StringIO

import pytest
import torch

from articulation3d_b200 import OptConfig, adapter, io, opt_utils, synth
from articulation3d_b200.axis import angle_offset_to_axis
from articulation3d_b200.tools import opt_arti

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 2021
SUMMARY = re.compile(r"^(\d+) video\(s\), (\d+) track\(s\): (\d+) track-frame x candidate evaluations in ")
LAUNCHERS = pytest.mark.parametrize("launcher", [
    pytest.param("nccl", marks=pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")),
    "one_gpu"])


def _descendants(pid):
    children = {}
    for d in os.listdir("/proc"):
        try:
            with open(f"/proc/{d}/stat") as f:
                children.setdefault(int(f.read().rsplit(")", 1)[1].split()[1]), []).append(int(d))
        except (OSError, ValueError, IndexError):
            continue
    out, todo = [], [pid]
    while todo:
        for c in children.get(todo.pop(), []):
            out.append(c)
            todo.append(c)
    return out


def torchrun(launcher, *args, timeout=900):
    """The tool on 2 ranks -> (return code, stdout, stderr).  torchrun starts every worker in a session of its
    own, so on a timeout the whole process tree is killed, not just the launcher."""
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join(p for p in (ROOT, env.get("PYTHONPATH")) if p)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nnodes", "1", "--nproc-per-node", "2",
           *(["-m", "articulation3d_b200.tools.opt_arti"] if launcher == "nccl" else
             [os.path.join(ROOT, "tests", "one_gpu_ranks.py")]), *map(str, args)]
    proc = subprocess.Popen(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                            start_new_session=True)
    try:
        out, err = proc.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        for p in _descendants(proc.pid) + [proc.pid]:
            try:
                os.kill(p, signal.SIGKILL)
            except ProcessLookupError:
                pass
        proc.communicate()
        raise
    return proc.returncode, out, err


def run_in_process(*args):
    buf = StringIO()
    with redirect_stdout(buf):
        opt_arti.main([str(a) for a in args])
    return buf.getvalue()


def write_gt(records, path):
    """COCO ground truth from the first detection of every frame, its rotation axis taken from the prediction
    (as test_gpu_adapter.py's AP test)."""
    images, anns = [], []
    for r in records:
        images.append({"id": r["image_id"], "width": 640, "height": 480})
        if not r["instances"]:
            continue
        ins = r["instances"][0]
        x, y, w, h = ins["bbox"]
        centre = torch.tensor([[x + w / 2, y + h / 2]], dtype=torch.float32)
        line = angle_offset_to_axis(torch.as_tensor(r["pred_rot_axis"][:1]).float(), centre)[0].tolist()
        cls = int(ins["category_id"])
        anns.append({"id": len(anns) + 1, "image_id": r["image_id"], "category_id": cls + 1, "bbox": [x, y, w, h],
                     "rot_axis": line if cls == 0 else None, "tran_axis": None, "normal": None})
    with open(path, "w") as f:
        json.dump({"images": images, "annotations": anns,
                   "categories": [{"id": 1, "name": "arti_rot"}, {"id": 2, "name": "arti_tran"}]}, f)


def same(a, b) -> bool:
    if isinstance(a, torch.Tensor):
        return isinstance(b, torch.Tensor) and a.dtype == b.dtype and torch.equal(a, b)
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(same(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return type(a) is type(b) and len(a) == len(b) and all(same(x, y) for x, y in zip(a, b))
    return type(a) is type(b) and bool(a == b)


def assert_same_outputs(want_dir, got_dir):
    files = sorted(os.listdir(want_dir))
    assert files and files == sorted(os.listdir(got_dir))
    for name in files:
        a, b = os.path.join(want_dir, name), os.path.join(got_dir, name)
        if name.endswith(".pth"):
            assert same(torch.load(a, weights_only=False), torch.load(b, weights_only=False)), name
        else:
            with open(a, "rb") as fa, open(b, "rb") as fb:
                assert fa.read() == fb.read(), name


@pytest.fixture(scope="module")
def one_gpu(tmp_path_factory):
    """5 synthetic videos (3 tracks x 14 frames: 3 + 2 on two ranks) optimised in-process on one GPU."""
    d = tmp_path_factory.mktemp("one_gpu")
    inp, gt = d / "pred.pth", d / "gt.json"
    run_in_process("--input", inp, "--output", d / "scratch", "--synthetic", 5, "--tracks", 3, "--frames", 14,
                   "--seed", SEED, "--device", DEV)
    write_gt(torch.load(inp, weights_only=False), gt)
    flags = ("--save-masks", "--save-obj", "--gt-json", gt)
    text = run_in_process("--input", inp, "--output", d / "out", "--seed", SEED, "--device", DEV, *flags)
    return {"input": inp, "out": d / "out", "flags": flags, "lines": text.splitlines()}


@LAUNCHERS
def test_sharded_run_equals_one_gpu_run(launcher, one_gpu, tmp_path):
    # the sharded run writes its own synthetic input (rank 0 writes, rank 1 waits): same seeds, same records
    rc, out, err = torchrun(launcher, "--input", tmp_path / "pred.pth", "--output", tmp_path / "out",
                            "--synthetic", 5, "--tracks", 3, "--frames", 14, "--seed", SEED, *one_gpu["flags"])
    assert rc == 0, err[-4000:]
    assert_same_outputs(one_gpu["out"], tmp_path / "out")
    lines = out.splitlines()
    want_ap = [l for l in one_gpu["lines"] if l.startswith("AP ")]
    assert len(want_ap) == 2 and [l for l in lines if l.startswith("AP ")] == want_ap
    summary = [l for l in lines if SUMMARY.match(l)]
    want = [SUMMARY.match(l).groups() for l in one_gpu["lines"] if SUMMARY.match(l)]
    assert len(summary) == 1 and summary[0].endswith(" on 2 GPUs")
    assert SUMMARY.match(summary[0]).groups() == want[0]
    assert want[0][0] == "5"


@LAUNCHERS
def test_more_ranks_than_videos(launcher, tmp_path):
    """1 video on 2 ranks: rank 1's block is empty; it joins the collectives and writes nothing."""
    inp = tmp_path / "pred.pth"
    run_in_process("--input", inp, "--output", tmp_path / "one", "--synthetic", 1, "--tracks", 3, "--frames", 14,
                   "--seed", SEED, "--device", DEV, "--save-obj")
    rc, out, err = torchrun(launcher, "--input", inp, "--output", tmp_path / "two", "--seed", SEED, "--save-obj")
    assert rc == 0, err[-4000:]
    assert_same_outputs(tmp_path / "one", tmp_path / "two")
    summary = [l for l in out.splitlines() if SUMMARY.match(l)]
    assert len(summary) == 1 and summary[0].startswith("1 video(s)") and summary[0].endswith(" on 2 GPUs")


@LAUNCHERS
def test_device_flag_refused_under_torchrun(launcher, one_gpu, tmp_path):
    rc, _, err = torchrun(launcher, "--input", one_gpu["input"], "--output", tmp_path / "out", "--device", "cuda:1")
    assert rc != 0
    assert "--device cannot be used under torchrun" in err
    assert not os.path.exists(tmp_path / "out")


def test_records_at_1024x768_use_the_scaled_camera(tmp_path):
    """The tool takes the camera from the records' frame size: its tracks equal the API's with
    OptConfig.scaled(1024, 768) and the same seeds."""
    cfg = OptConfig.scaled(1024, 768)
    records = []
    for v in range(2):
        preds, _ = synth.make_video(SEED + v, 3, 14, cfg)
        records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000, device=DEV)
    inp, out = tmp_path / "pred.pth", tmp_path / "out"
    torch.save(records, inp)
    run_in_process("--input", inp, "--output", out, "--seed", SEED, "--device", DEV)
    groups = adapter.group_by_video(records)
    videos = [(p, opt_utils.track_planes(p, cfg)) for p in
              (io.records_to_preds(recs, masks="rle") for recs in groups.values())]
    opt_utils.optimize_videos(videos, [SEED + i for i in range(len(videos))], cfg=cfg, device=DEV)
    for vid, (_, planes) in zip(groups, videos):
        with open(out / f"{vid}_tracks.json") as f:
            got = json.load(f)
        assert got == json.loads(json.dumps(io.tracks_summary(planes)))
        assert any(t["has_rot"] for t in got)
