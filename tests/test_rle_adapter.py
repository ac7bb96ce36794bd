"""CPU tests of the COCO RLE codec and the per-frame adapter (no GPU)."""
import numpy as np
import pytest
import torch

from articulation3d_b200 import adapter, rle
from oracle import restated


@pytest.mark.parametrize("shape", [(480, 640), (5, 7), (1, 1), (33, 100)])
def test_rle_round_trip_and_oracle_agree(shape):
    rng = np.random.RandomState(shape[0])
    h, w = shape
    cases = [np.zeros(shape, bool), np.ones(shape, bool), rng.rand(h, w) < 0.5, rng.rand(h, w) < 0.02]
    m = np.zeros(shape, bool)
    m[h // 4: h // 2 + 1, w // 3: w // 2 + 1] = True
    cases.append(m)
    for m in cases:
        r = rle.encode(m)
        assert r["size"] == [h, w] and isinstance(r["counts"], bytes)
        assert all(48 <= c < 48 + 64 for c in r["counts"])              # printable ASCII, 6 bits per char
        c = rle.rle_counts(r)
        assert int(c.astype(np.int64).sum()) == h * w
        assert rle.counts_to_string(c) == r["counts"]
        assert np.array_equal(rle.decode(r).astype(bool), m)
        assert np.array_equal(restated.rle_decode(r).astype(bool), m)     # independent decoder
        assert np.array_equal(rle.decode({"size": [h, w], "counts": c.tolist()}).astype(bool), m)


def test_rle_varint_known_structure():
    # counts < 16 take one character (value + 48); the third count onwards is a signed delta
    assert rle.counts_to_string([3, 5]) == bytes([48 + 3, 48 + 5])
    assert rle.string_to_counts(bytes([48 + 3, 48 + 5])).tolist() == [3, 5]
    c = [0, 300000, 5, 7, 100000, 1, 1195]
    assert rle.string_to_counts(rle.counts_to_string(c)).tolist() == c
    # column-major: a single pixel at (row 1, col 0) of a 3x2 mask is run [1, 1, 4]
    m = np.zeros((3, 2), bool)
    m[1, 0] = True
    assert rle.rle_counts(rle.encode(m)).tolist() == [1, 1, 4]
    with pytest.raises(ValueError):
        rle.decode({"size": [3, 2], "counts": [1, 1]})


def test_create_instances_contract():
    h, w = 48, 64
    m = np.zeros((h, w), bool)
    m[10:20, 5:30] = True
    dets = [{"score": 0.9, "bbox": [5, 10, 25, 10], "category_id": 0, "segmentation": rle.encode(m)},
            {"score": 0.5, "bbox": [0, 0, 4, 4], "category_id": 1, "segmentation": rle.encode(~m)},
            {"score": 0.8, "bbox": [1, 2, 3, 4], "category_id": 1, "segmentation": rle.encode(~m)}]
    planes = torch.arange(9.).reshape(3, 3)
    rot = torch.arange(9.).reshape(3, 3) + 10
    tran = torch.arange(6.).reshape(3, 2)
    inst = adapter.create_instances(dets, (h, w), planes, rot, tran, conf_threshold=0.7)
    assert len(inst) == 2 and inst.pred_classes.tolist() == [0, 1]
    assert inst.pred_boxes.tensor.tolist() == [[5, 10, 30, 20], [1, 2, 4, 6]]          # XYWH -> XYXY
    assert torch.equal(inst.pred_planes, planes[[0, 2]]) and torch.equal(inst.pred_rot_axis, rot[[0, 2]])
    assert inst.pred_masks.dtype == torch.float32 and inst.pred_masks.shape == (2, h, w)
    assert np.array_equal(inst.pred_masks[0].numpy() > 0.5, m)
    lazy = adapter.create_instances(dets, (h, w), planes, rot, tran, masks="rle")
    assert not lazy.has("pred_masks") and len(lazy.pred_rle) == 2
    # ADVICE r1: two shots of the same YouTube id are two videos; frames are ordered by their offset
    recs = [{"file_name": "a/abcdefghijk_1_20_15.png"}, {"file_name": "abcdefghijk_1_20_5.png"},
            {"file_name": "zzzzzzzzzzz_0_0_5.png"}, {"file_name": "x/abcdefghijk_2_300_7.png"},
            {"file_name": "x/abcdefghijk_2_300_6.png"}, {"file_name": "abc_def_hij_3_4_0.png"}]
    groups = adapter.group_by_video(recs)
    assert list(groups) == ["abcdefghijk_1_20", "zzzzzzzzzzz_0_0", "abcdefghijk_2_300", "abc_def_hij_3_4"]
    assert [r["file_name"] for r in groups["abcdefghijk_1_20"]] == ["abcdefghijk_1_20_5.png", "a/abcdefghijk_1_20_15.png"]
    assert [r["file_name"][-5:] for r in groups["abcdefghijk_2_300"]] == ["6.png", "7.png"]


def test_ray_table_matches_reference_loop_on_a_subgrid():
    """The vectorised table is the reference's double loop bit for bit at every frame size the tool and the depth
    override use it at: odd and 1-pixel sizes, rows wider than 1024."""
    for h, w in ((48, 64), (37, 1057), (1, 1), (768, 1024)):
        a = adapter.get_K_inv_dot_xy_1(h, w)
        b = restated.get_K_inv_dot_xy_1(h, w)
        assert a.shape == (3, h, w)
        assert np.array_equal(a, b), (h, w)


def test_native_string_decoder_equals_python_decoder():
    """a3d_host_rle_counts (host helper of liba3d.so) against rle.string_to_counts on structured, dense-random and
    degenerate masks, str and bytes inputs, an empty string; malformed strings are refused."""
    from articulation3d_b200 import _lib
    rng = np.random.RandomState(3)
    H, W = 120, 160
    masks = []
    m = np.zeros((H, W), bool); masks.append(m.copy())
    m[:] = True; masks.append(m.copy())
    m[:] = False; m[20:90, 30:100] = True; masks.append(m.copy())
    masks.append(rng.rand(H, W) < 0.5)
    masks.append(rng.rand(H, W) < 0.01)
    m = np.zeros((H, W), bool); m[0, 0] = m[-1, -1] = True; masks.append(m.copy())
    m = np.zeros((H, W), bool); m[:, ::2] = True; masks.append(m.copy())          # equal long runs: zero differences
    rls = [rle.encode(x) for x in masks]
    strings = [r["counts"] if i % 2 else r["counts"].decode("ascii") for i, r in enumerate(rls)] + [b""]
    flat, begin, sums = rle.strings_to_counts(strings)
    assert flat.dtype == np.uint32 and begin[0] == 0 and begin[-1] == len(flat)
    for i, r in enumerate(rls):
        assert np.array_equal(flat[begin[i]:begin[i + 1]], rle.string_to_counts(r["counts"])), i
        assert sums[i] == H * W
    assert begin[-2] == begin[-1] and sums[-1] == 0
    big = np.zeros((900, 1200), bool); big[7:880, 5:1190] = True                    # counts beyond 2^15 / 2^20
    f, b, s = rle.strings_to_counts([rle.encode(big)["counts"]])
    assert np.array_equal(f, rle.string_to_counts(rle.encode(big)["counts"])) and s[0] == 900 * 1200
    f, b, s = rle.strings_to_counts([])
    assert len(f) == 0 and list(b) == [0]
    with pytest.raises(_lib.A3DError):
        rle.strings_to_counts([b"0P"])                                              # continuation bit on the last character
