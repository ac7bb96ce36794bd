"""GPU tests of the COCO RLE encoder (a3d_rle_count_runs / a3d_bits_to_rle, engine.bits_to_rle, rle.encode_many) and
of everything that saves masks through it: the records writer, RegMasks.to_rle and the tools' --save-masks.  The
oracle is rle.encode on the host, compared byte for byte; encoded masks are also decoded back on the device."""
import json
import os
import random

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, io, opt_utils, rle, synth
from articulation3d_b200.structures import Boxes, Instances
from articulation3d_b200.tools import inference, opt_arti
from oracle import restated
from tests import golden_util

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SHAPES = [(1, 1), (1, 1000), (1000, 1), (5, 7), (33, 100), (480, 640), (768, 1024), (1025, 1023), (2048, 2048)]


def _structured(H, W, seed):
    """Boundary cases of the column-major run structure for an H x W frame."""
    rng = np.random.RandomState(seed)
    out = {"empty": np.zeros((H, W), bool), "full": np.ones((H, W), bool)}
    m = np.zeros((H, W), bool); m[0, 0] = True; out["first"] = m
    m = np.zeros((H, W), bool); m[-1, -1] = True; out["last"] = m
    m = np.zeros((H, W), bool)
    for x in (31, 32, 63, 64, W - 1):                    # word boundaries and the last column
        if x < W:
            m[0, x] = m[H - 1, x] = m[H // 2, x] = True
    out["word_edges"] = m
    if W >= 2:
        m = np.zeros((H, W), bool); m[:, W // 2 - 1: W // 2 + 1] = True; out["two_columns"] = m
        m = np.zeros((H, W), bool); m[H - 1, W // 2 - 1] = m[0, W // 2] = True; out["wrap"] = m
        m = np.zeros((H, W), bool); m[:, ::2] = True; out["stripes"] = m
    out["checker"] = (np.add.outer(np.arange(H), np.arange(W)) % 2) == 0
    out["dense"] = rng.rand(H, W) < 0.5
    out["sparse"] = rng.rand(H, W) < 0.01
    m = np.zeros((H, W), bool); m[H // 5: 4 * H // 5 + 1, W // 3: W // 2 + 1] = True; out["door"] = m
    return out


def _decode_matches(rles, masks, H, W):
    """Decode through engine.rle_to_pool and compare the packed words with the packed masks."""
    if H * _lib.pitch_words(W) * 4 > 200 * 1024:        # rle_to_pool decodes frames that fit shared memory
        return
    pool = engine.rle_to_pool(rles, H, W, DEV)
    want = engine.pack_masks(torch.from_numpy(np.ascontiguousarray(masks != 0)).to(DEV)).bits
    assert torch.equal(pool.bits, want)


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_encode_many_equals_host_encoder(shape):
    H, W = shape
    cases = _structured(H, W, H * 7 + W)
    names = list(cases)
    masks = np.stack([cases[k] for k in names])
    want = [rle.encode(m) for m in masks]
    got = rle.encode_many(masks, device=DEV)                                  # bool, from the host
    for k, g, w in zip(names, got, want):
        assert g == w, k
    if H % 2 == 1:                                                           # a boundary at every pixel
        assert len(rle.rle_counts(got[names.index("checker")])) == H * W + 1
    _decode_matches(got, masks, H, W)
    if H * W <= 1 << 20:
        assert rle.encode_many(torch.from_numpy(masks).to(DEV)) == want    # bool, already on the device
        assert rle.encode_many(masks.astype(np.uint8) * 7, device=DEV) == want


def test_encode_many_float_inputs_use_nonzero():
    """fp32 masks are tested with != 0, as rle.encode does: NaN and denormals are set, -0.0 is not."""
    rng = np.random.RandomState(5)
    H, W = 37, 70
    m = rng.choice(np.array([0.0, -0.0, 1.0, np.nan, 1e-40, -1e-45, 0.25, -3.0], np.float32), size=(6, H, W))
    want = [rle.encode(x) for x in m]
    assert rle.encode_many(m, device=DEV) == want
    assert rle.encode_many(torch.from_numpy(m).to(DEV)) == want
    assert rle.encode_many(torch.from_numpy(m), device=torch.device(DEV)) == want


def test_encode_many_chunks_and_empty(monkeypatch):
    monkeypatch.setattr(rle, "ENCODE_CHUNK", 3)
    rng = np.random.RandomState(2)
    m = (rng.rand(10, 20, 45) < 0.3).astype(np.float32)
    assert rle.encode_many(m, device=DEV) == [rle.encode(x) for x in m]
    assert rle.encode_many(np.zeros((0, 4, 4), np.float32), device=DEV) == []


def test_bits_to_rle_index_and_many_masks(monkeypatch):
    monkeypatch.setenv("A3D_WS_POISON", "1")
    rng = np.random.RandomState(9)
    masks = rng.rand(7, 50, 90) < 0.2
    bits = engine.pack_masks(torch.from_numpy(masks).to(DEV)).bits
    index = torch.tensor([3, 3, 0, 6, 1, 3], dtype=torch.int32, device=DEV)
    counts, begin = engine.bits_to_rle(bits, 50, 90, index)
    assert begin.dtype == np.int64 and counts.dtype == np.uint32 and len(begin) == 7
    for i, k in enumerate(index.tolist()):
        assert counts[begin[i]:begin[i + 1]].tolist() == rle.rle_counts(rle.encode(masks[k])).tolist()
    assert [r["counts"] for r in rle.bits_to_rles(bits, 50, 90, index)] == [rle.encode(masks[k])["counts"]
                                                                            for k in index.tolist()]
    counts, begin = engine.bits_to_rle(bits[:0], 50, 90)
    assert len(counts) == 0 and begin.tolist() == [0]
    # more masks than the 65535 blocks of a grid's y / z dimension
    many = rng.rand(70000, 4, 4) < 0.5
    assert rle.encode_many(many, device=DEV) == [rle.encode(x) for x in many]


def test_abi_writes_exactly_its_range_and_checks_arguments():
    lib = _lib.load()
    rng = np.random.RandomState(4)
    H, W = 45, 77
    masks = rng.rand(5, H, W) < 0.3
    masks[2] = False
    masks[3, 0, 0] = True
    bits = engine.pack_masks(torch.from_numpy(masks).to(DEV)).bits
    want = [rle.rle_counts(rle.encode(m)) for m in masks]
    s = torch.cuda.current_stream().cuda_stream
    runs = torch.full((5 + 4,), -0x5454545454545455, dtype=torch.int64, device=DEV)      # 0xAB.. bytes + guard
    assert lib.a3d_rle_count_runs(bits.data_ptr(), None, 5, H, W, runs.data_ptr(), s) == 0
    r = runs.cpu()
    assert r[:5].tolist() == [len(c) for c in want] and r[5:].eq(-0x5454545454545455).all()
    begin = torch.zeros(6, dtype=torch.int64, device=DEV)
    begin[1:] = torch.cumsum(runs[:5], 0)
    total = int(begin[-1])
    out = torch.full(((total + 16) * 4,), 0xAB, dtype=torch.uint8, device=DEV)          # runs + a 16-count guard
    assert lib.a3d_bits_to_rle(bits.data_ptr(), None, 5, H, W, begin.data_ptr(), out.data_ptr(), s) == 0
    o = out.cpu()
    got = o[:total * 4].numpy().view(np.uint32)
    assert np.array_equal(got, np.concatenate(want)) and o[total * 4:].eq(0xAB).all()
    # bad arguments: A3D_EINVAL; frames of 2^31 pixels or more: A3D_ELIMIT before anything is touched
    for rc in (lib.a3d_rle_count_runs(bits.data_ptr(), None, -1, H, W, runs.data_ptr(), s),
               lib.a3d_rle_count_runs(bits.data_ptr(), None, 5, 0, W, runs.data_ptr(), s),
               lib.a3d_rle_count_runs(bits.data_ptr(), None, 5, H, -3, runs.data_ptr(), s),
               lib.a3d_rle_count_runs(None, None, 5, H, W, runs.data_ptr(), s),
               lib.a3d_rle_count_runs(bits.data_ptr(), None, 5, H, W, None, s),
               lib.a3d_bits_to_rle(bits.data_ptr(), None, 5, H, W, None, out.data_ptr(), s),
               lib.a3d_bits_to_rle(bits.data_ptr(), None, 5, H, W, begin.data_ptr(), None, s)):
        assert rc == -1
    assert lib.a3d_rle_count_runs(None, None, 0, H, W, None, s) == 0
    assert lib.a3d_rle_count_runs(None, None, 0, 1, 0x7fffffff, None, s) == 0              # 2^31 - 1 pixels: allowed
    for h, w in ((1 << 16, 1 << 15), (46341, 46341), (2, 0x7fffffff)):
        assert lib.a3d_rle_count_runs(None, None, 1, h, w, None, s) == -3
        assert f"{h}x{w}".encode() in lib.a3d_last_error_string()
        assert lib.a3d_bits_to_rle(None, None, 1, h, w, None, None, s) == -3
    torch.cuda.synchronize()


def _golden(name):
    z = golden_util.load(name)
    return z, golden_util.arrays_to_preds(z, Instances, Boxes), int(z["image_size"][1])


@pytest.mark.parametrize("case", golden_util.golden_cases())
def test_reg_masks_to_rle_equal_reference_masks(case):
    """RegMasks.to_rle() of every fitted track == rle.encode of the reference's own registered masks."""
    z, preds, W = _golden(case)
    random.seed(int(z["seed"]))
    planes = opt_utils.track_planes(preds)
    opt_utils.optimize_planes(preds, planes, '3dc', device=DEV)
    _check_reg_masks(planes, z, W)


def _check_reg_masks(planes, z, W):
    checked = 0
    for cat in ("trans", "rot"):
        for i, p in enumerate(planes[cat]):
            if not p["has_rot"]:
                continue
            gold = golden_util.unpack_bits(z[f"{cat}{i}_reg_masks"], W)
            rles = p["reg_masks"].to_rle()
            assert list(rles) == z[f"{cat}{i}_reg_frames"].tolist()
            assert not p["reg_masks"]._cache
            for j, f in enumerate(rles):
                assert rles[f] == rle.encode(gold[j]), (cat, i, f)
                checked += 1
    assert checked > 0


def test_reg_masks_to_rle_through_worker_streams(monkeypatch):
    """The same through optimize_videos with two pipeline workers: the packed masks were made on the workers'
    streams and are encoded on the caller's."""
    monkeypatch.setenv("A3D_PIPELINE_WORKERS", "2")
    loaded = [_golden(c) for c in golden_util.golden_cases()]
    videos = [(preds, opt_utils.track_planes(preds)) for _, preds, _ in loaded]
    opt_utils.optimize_videos(videos, [int(z["seed"]) for z, _, _ in loaded], device=DEV)
    for (z, _, W), (_, planes) in zip(loaded, videos):
        _check_reg_masks(planes, z, W)


def test_preds_to_records_on_device_equal_host():
    preds, _ = synth.make_video(2020, 4, 120)
    host = io.preds_to_records(preds, video_id="v_0_0", start_image_id=7)
    dev = io.preds_to_records(preds, video_id="v_0_0", start_image_id=7, device=DEV)
    assert len(host) == len(dev) == 120
    for a, b in zip(host, dev):
        assert a["instances"] == b["instances"]
        assert all(isinstance(i["segmentation"]["counts"], bytes) for i in b["instances"])
        for k in ("pred_plane", "pred_rot_axis", "pred_tran_axis"):
            assert torch.equal(a[k], b[k])
        assert {k: v for k, v in a.items() if k != "instances" and not torch.is_tensor(v)} == \
            {k: v for k, v in b.items() if k != "instances" and not torch.is_tensor(v)}


def _tracks(out_dir, vid="synthetic00_0_0"):
    with open(os.path.join(out_dir, f"{vid}_tracks.json")) as f:
        return json.load(f)


def _assert_segmentations(tracks, planes_o, H, W):
    order = [p for cat in ("trans", "rot") for p in planes_o[cat]]
    assert len(tracks) == len(order)
    seen = 0
    for t, p in zip(tracks, order):
        if not t["has_rot"]:
            continue
        for e in t["angle_track"]:
            seg = e["segmentation"]
            assert seg["size"] == [H, W] and isinstance(seg["counts"], str)
            got = rle.decode(seg).astype(bool)
            assert np.array_equal(got, np.asarray(p["reg_masks"][e["frame"]]) > 0.5), e["frame"]
            seen += 1
    assert seen > 0


def test_inference_tool_save_masks(tmp_path):
    base = ["--frames", "30", "--tracks", "3", "--seed", "2020"]
    inference.main(["--output", str(tmp_path / "m")] + base + ["--save-masks"])
    inference.main(["--output", str(tmp_path / "p")] + base)
    with_masks, plain = _tracks(tmp_path / "m"), _tracks(tmp_path / "p")
    assert "segmentation" not in json.dumps(plain)
    stripped = json.loads(json.dumps(with_masks))
    for t in stripped:
        for e in t.get("angle_track", []):
            del e["segmentation"]
    assert stripped == plain
    preds, _ = synth.make_video(2020, 3, 30, OptConfig())
    random.seed(2020)
    planes_o = restated.track_planes(preds)
    restated.optimize_planes(preds, planes_o, "3dc")
    _assert_segmentations(with_masks, planes_o, 480, 640)


def test_opt_arti_synthetic_save_masks(tmp_path):
    inp = str(tmp_path / "in.pth")
    opt_arti.main(["--input", inp, "--output", str(tmp_path / "o"), "--synthetic", "2", "--tracks", "3",
                   "--frames", "30", "--save-masks"])
    host_records = []
    for v in range(2):
        preds, _ = synth.make_video(2020 + v, 3, 30)
        host_records += io.preds_to_records(preds, video_id=f"synthetic{v:02d}_0_0", start_image_id=v * 10000)
    saved = torch.load(inp, weights_only=False)
    assert [r["instances"] for r in saved] == [r["instances"] for r in host_records]
    from articulation3d_b200 import adapter
    groups = adapter.group_by_video(adapter.load_predictions(inp))
    for v, (vid, recs) in enumerate(groups.items()):
        preds = io.records_to_preds(recs, conf_threshold=0.7, masks="dense")
        random.seed(2020 + v)
        planes_o = restated.track_planes(preds)
        restated.optimize_planes(preds, planes_o, "3dc")
        _assert_segmentations(_tracks(tmp_path / "o", vid), planes_o, 480, 640)
