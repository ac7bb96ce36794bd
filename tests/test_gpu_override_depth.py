"""``adapter.override_depth_records`` (depth streamed through the device in chunks) against
``override_depth_batch`` bit for bit and against the reference's ``override_depth``; memory-mapped input, the
device-memory bound, the synthetic depth's self-check, and ``tools.opt_arti --override-depth`` against the API
sequence, on one GPU and under torchrun."""
import copy
import hashlib
import os
import re

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, adapter, io, opt_utils, rle, synth
from oracle import restated
from tests.test_gpu_opt_arti_sharded import LAUNCHERS, assert_same_outputs, run_in_process, torchrun, write_gt

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 2022
OVERRIDE = re.compile(r"^override-depth: (\d+) frame\(s\), (\d+) instance\(s\), ([0-9.]+) MB of depth in ")


def _cfg(H, W):
    return OptConfig() if (H, W) == (480, 640) else OptConfig.scaled(W, H)


def _records(H, W, videos=2, frames=10, seed=7):
    """Synthetic records with random depth, plus the edge cases: a frame with no instance, an empty mask and a
    full-frame mask (each with a plane of its own)."""
    cfg = _cfg(H, W)
    g = torch.Generator().manual_seed(seed)
    records = []
    for v in range(videos):
        preds, _ = synth.make_video(seed + v, 3, frames, cfg, kinds=[0, 1, 0])
        depths = 0.5 + 3 * torch.rand(frames, H, W, generator=g)
        records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                       device=DEV, depths=depths)
    r = records[3]
    for m in (np.zeros((H, W), bool), np.ones((H, W), bool)):
        r["instances"].append(dict(r["instances"][0], segmentation=rle.encode(m)))
    r["pred_plane"] = torch.cat([r["pred_plane"], torch.tensor([[0.3, 1.0, -0.2], [-0.1, 2.0, 0.4]])])
    r = records[-2]
    r["instances"], r["pred_plane"] = [], torch.zeros(0, 3)
    return records


def _batch(records):
    recs = copy.deepcopy(records)
    depths = torch.stack([r["pred_depth"] for r in recs]).to(DEV)
    return adapter.override_depth_batch(recs, depths=depths)


@pytest.mark.parametrize("H,W", [(480, 640), (768, 1024)])
@pytest.mark.parametrize("chunk_frames", [1, 7, None])
def test_records_equal_batch_bit_for_bit(H, W, chunk_frames):
    records = _records(H, W)
    want = _batch(records)
    inputs = [r["pred_plane"] for r in records]
    want_inputs = [p.clone() for p in inputs]
    for p in want_inputs:                                   # the batch path's in-place swap of the input tensor
        p[:, [1, 2]] = p[:, [2, 1]]
        p[:, 1] = -p[:, 1]
    chunk = (1 << 40) if chunk_frames is None else chunk_frames * H * W * 4
    out = adapter.override_depth_records(records, DEV, chunk_bytes=chunk)
    assert out is records
    for a, b in zip(records, want):
        assert a["pred_plane"].shape == b["pred_plane"].shape
        assert torch.equal(a["pred_plane"].view(torch.int32), b["pred_plane"].view(torch.int32)), a["file_name"]
    for p, q in zip(inputs, want_inputs):
        assert torch.equal(p.view(torch.int32), q.view(torch.int32))
    r = records[3]
    assert torch.equal(r["pred_plane"][-2], torch.tensor([0.3, 1.0, -0.2]))          # the empty mask keeps it
    assert not torch.equal(r["pred_plane"][-1], torch.tensor([-0.1, 2.0, 0.4]))
    assert not torch.equal(records[0]["pred_plane"], _records(H, W)[0]["pred_plane"])


def test_records_match_reference_at_768x1024():
    H, W = 768, 1024
    records = _records(H, W, videos=1, frames=4)
    want = copy.deepcopy(records)
    adapter.override_depth_records(records, DEV, chunk_bytes=2 * H * W * 4)
    rays = torch.FloatTensor(adapter.get_K_inv_dot_xy_1(H, W))
    for r, w in zip(records, want):
        ref = restated.override_depth(rays * w["pred_depth"], w)["pred_plane"]
        np.testing.assert_allclose(r["pred_plane"].numpy(), ref.numpy(), rtol=1e-4, atol=1e-6)


MIXED = [(480, 640)] * 3 + [(29, 1057)] * 2 + [None] + [(480, 640)] * 2 + [(768, 1024)]


def _mixed_records(seed=3):
    """Records of changing frame sizes (``MIXED``; None: a 480x640 record without instances) with edge and blob
    masks, random planes and random fp32 depth; plus each record's masks."""
    from tests.test_gpu_plane_offsets import edge_masks
    rng = np.random.RandomState(seed)
    records, masks = [], []
    for t, size in enumerate(MIXED):
        H, W = size or (480, 640)
        e = edge_masks(H, W, rng)
        m = e[rng.permutation(len(e))[:4 + t % 3]] if size else e[:0]
        records.append({"file_name": f"mixed_{t}.png", "instances": [{"segmentation": rle.encode(x)} for x in m],
                        "pred_plane": torch.from_numpy(rng.normal(size=(len(m), 3)).astype(np.float32)),
                        "pred_depth": torch.from_numpy(rng.uniform(0.5, 4, (H, W)).astype(np.float32))})
        masks.append(m)
    return records, masks


@pytest.mark.parametrize("chunk_bytes", [1, 2 * 768 * 1024 * 4, 1 << 40], ids=["1_frame", "2_largest", "all"])
def test_records_of_mixed_sizes(chunk_bytes):
    """Chunks end where the frame size changes: the planes are bit-equal to ``override_depth_batch`` of each
    same-size group and within the bound of the float64 reference (tests/test_gpu_plane_offsets.py), whatever
    the chunk size."""
    from tests.test_gpu_plane_offsets import assert_planes, reference_planes
    records, masks = _mixed_records()
    inputs = [r["pred_plane"].clone() for r in records]
    groups = {}
    for i, r in enumerate(records):
        if r["instances"]:
            groups.setdefault(tuple(r["pred_depth"].shape), []).append(i)
    want = {}
    for (H, W), idx in groups.items():
        recs = [dict(records[i], pred_plane=inputs[i].clone()) for i in idx]
        out = adapter.override_depth_batch(recs, depths=torch.stack([r["pred_depth"] for r in recs]).to(DEV))
        want.update({i: r["pred_plane"] for i, r in zip(idx, out)})
        rays = adapter.get_K_inv_dot_xy_1(H, W).astype(np.float32)
        frame_of = np.concatenate([np.full(len(masks[i]), k) for k, i in enumerate(idx)])
        ref = reference_planes(torch.cat([inputs[i] for i in idx]), np.concatenate([masks[i] for i in idx]),
                               frame_of, rays, np.stack([records[i]["pred_depth"].numpy() for i in idx]))
        assert_planes(torch.cat([want[i] for i in idx]), ref, f"{H}x{W}")
    adapter.override_depth_records(records, DEV, chunk_bytes=chunk_bytes)
    for i, r in enumerate(records):
        if i in want:
            assert torch.equal(r["pred_plane"].view(torch.int32), want[i].view(torch.int32)), r["file_name"]
        else:
            assert r["pred_plane"].shape == (0, 3)


def test_memory_mapped_file_is_unchanged(tmp_path):
    path = str(tmp_path / "pred.pth")
    torch.save(_records(480, 640), path)
    digest = hashlib.sha256(open(path, "rb").read()).hexdigest()
    mapped = adapter.load_predictions(path, mmap=True)
    read = adapter.load_predictions(path)
    adapter.override_depth_records(mapped, DEV, chunk_bytes=3 * 480 * 640 * 4)
    adapter.override_depth_records(read, DEV)
    assert hashlib.sha256(open(path, "rb").read()).hexdigest() == digest
    for a, b in zip(mapped, read):
        assert torch.equal(a["pred_plane"].view(torch.int32), b["pred_plane"].view(torch.int32))


def test_device_memory_is_bounded_by_the_chunk():
    H, W = 480, 640
    records = _records(H, W, videos=3, frames=20)
    chunk = 4 * H * W * 4
    adapter.override_depth_records(copy.deepcopy(records[:1]), DEV)       # rays of this size are built and cached
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    adapter.override_depth_records(records, DEV, chunk_bytes=chunk)
    growth = torch.cuda.max_memory_allocated() - base
    per_frame = max(len(r["instances"]) for r in records)
    pool = 4 * per_frame * H * _lib.pitch_words(W) * 4
    total_depth = len(records) * H * W * 4
    bound = 2 * chunk + pool + (1 << 20)                   # + counts, boxes, RLE runs and results of one chunk
    assert growth <= bound < total_depth / 4, (growth, bound, total_depth)


def test_synthetic_depth_gives_back_the_true_planes():
    """Records holding the scene's true planes come back within 1e-4 for every instance whose plane lies in front
    of the camera over its whole mask (no mask pixel of it got the background depth)."""
    checked = 0
    for seed in (2020, 2021):
        preds, scene = synth.make_video(seed, 4, 12)
        depths = synth.render_depths(scene, background=50.0)
        records = io.preds_to_records(preds, device=DEV, depths=depths)
        true = synth.scene_pred_planes(scene)
        for t, r in enumerate(records):
            r["pred_plane"] = true[:, t].clone()
        adapter.override_depth_records(records, DEV, chunk_bytes=5 * 480 * 640 * 4)
        for t, (p, r) in enumerate(zip(preds, records)):
            for k, m in enumerate(p.pred_masks):
                m = m > 0.5
                if bool(m.any()) and bool((depths[t][m] < 50.0).all()):
                    np.testing.assert_allclose(r["pred_plane"][k].numpy(), true[k, t].numpy(), rtol=1e-4, atol=1e-6)
                    checked += 1
    assert checked >= 48


def _api(inp, out_dir, override, seed=SEED):
    """The tool's sequence through the API: load -> [override_depth_records] -> records_to_preds -> track_planes
    -> optimize_videos (seed + i) -> save_results."""
    groups = adapter.group_by_video(adapter.load_predictions(str(inp)))
    if override:
        adapter.override_depth_records([r for recs in groups.values() for r in recs], DEV)
    videos = []
    for recs in groups.values():
        preds = io.records_to_preds(recs, masks="rle")
        videos.append((preds, opt_utils.track_planes(preds, OptConfig())))
    outs = opt_utils.optimize_videos(videos, [seed + i for i in range(len(videos))], cfg=OptConfig(), device=DEV)
    for (vid, recs), out, (_, planes) in zip(groups.items(), outs, videos):
        io.save_results(str(out_dir), vid, io.opt_preds_to_records(out, recs), planes, masks=True)


def _synthetic_records(n, tracks, frames, seed=SEED):
    records = []
    for v in range(n):
        preds, scene = synth.make_video(seed + v, tracks, frames)
        records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000,
                                       device=DEV, depths=synth.render_depths(scene))
    return records


@pytest.fixture(scope="module")
def tool_run(tmp_path_factory):
    """``--synthetic 3 --synthetic-depth --override-depth --save-masks --gt-json`` in-process on one GPU."""
    d = tmp_path_factory.mktemp("override_tool")
    gt = d / "gt.json"
    write_gt(_synthetic_records(3, 3, 14), gt)
    flags = ("--override-depth", "--save-masks", "--gt-json", gt)
    text = run_in_process("--input", d / "pred.pth", "--output", d / "out", "--synthetic", 3, "--synthetic-depth",
                          "--tracks", 3, "--frames", 14, "--seed", SEED, "--device", DEV, *flags)
    return {"dir": d, "input": d / "pred.pth", "out": d / "out", "gt": gt, "flags": flags,
            "lines": text.splitlines()}


def test_tool_equals_api_sequence(tool_run, tmp_path):
    d = tool_run["dir"]
    want = _synthetic_records(3, 3, 14)
    got = torch.load(tool_run["input"], weights_only=False)
    assert [torch.equal(a["pred_depth"], b["pred_depth"]) for a, b in zip(got, want)] == [True] * len(want)
    _api(tool_run["input"], tmp_path / "api", override=True)
    assert_same_outputs(tmp_path / "api", tool_run["out"])
    lines = tool_run["lines"]
    m = [OVERRIDE.match(l) for l in lines if OVERRIDE.match(l)]
    n_inst = sum(len(r["instances"]) for r in want)
    assert len(m) == 1 and m[0].groups()[:2] == (str(len(want)), str(n_inst))
    assert len([l for l in lines if l.startswith("AP ")]) == 2

    # without the flag: the API sequence without the override, and other planes
    run_in_process("--input", tool_run["input"], "--output", d / "plain", "--seed", SEED, "--device", DEV,
                   "--save-masks")
    _api(tool_run["input"], tmp_path / "api_plain", override=False)
    assert_same_outputs(tmp_path / "api_plain", d / "plain")
    vid = "synthetic00_0_0"
    a = torch.load(d / "plain" / f"{vid}_predictions_opt.pth", weights_only=False)
    b = torch.load(tool_run["out"] / f"{vid}_predictions_opt.pth", weights_only=False)
    assert sum(not torch.equal(x["pred_plane"], y["pred_plane"]) for x, y in zip(a, b)) >= len(a) - 1


def test_tool_refuses_records_without_depth(tmp_path):
    inp = tmp_path / "pred.pth"
    run_in_process("--input", inp, "--output", tmp_path / "w", "--synthetic", 1, "--tracks", 2, "--frames", 6,
                   "--seed", SEED, "--device", DEV)
    with pytest.raises(ValueError, match="pred_depth"):
        run_in_process("--input", inp, "--output", tmp_path / "out", "--device", DEV, "--override-depth")
    assert not os.path.exists(tmp_path / "out")


@LAUNCHERS
def test_sharded_override_equals_one_gpu_run(launcher, tool_run, tmp_path):
    rc, out, err = torchrun(launcher, "--input", tool_run["input"], "--output", tmp_path / "out", "--seed", SEED,
                            *tool_run["flags"])
    assert rc == 0, err[-4000:]
    assert_same_outputs(tool_run["out"], tmp_path / "out")
    lines = out.splitlines()
    want_ap = [l for l in tool_run["lines"] if l.startswith("AP ")]
    assert len(want_ap) == 2 and [l for l in lines if l.startswith("AP ")] == want_ap
    got = [l for l in lines if OVERRIDE.match(l)]
    want = [OVERRIDE.match(l).groups() for l in tool_run["lines"] if OVERRIDE.match(l)]
    assert len(got) == 1 and got[0].endswith(" on 2 GPUs") and OVERRIDE.match(got[0]).groups() == want[0]
