"""CPU tests of the clip renderer: the numpy restatement of a3d_render on hand-made known answers, the draw lists
render.draw_lists builds, and engine.render's argument checks (no GPU)."""
import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, axis, engine, render, synth
from tests import render_ref


def _lists(layers=(), segs=(), T=1):
    lay = np.array(list(layers), dtype=_lib.LAYER_DTYPE)
    sg = np.array(list(segs), dtype=_lib.SEGMENT_DTYPE)
    lb = np.zeros(T + 1, np.int64)
    sb = np.zeros(T + 1, np.int64)
    lb[1:] = len(lay)
    sb[1:] = len(sg)
    return lay, lb, sg, sb


def _seg_pixels(H, W, *seg):
    return set(zip(*np.nonzero(render_ref.segment_cover(H, W, *seg))[::-1]))      # {(x, y)}


def test_outline_of_a_filled_square_is_its_ring():
    m = np.zeros((7, 7), bool)
    m[2:5, 2:5] = True
    ring = m.copy()
    ring[3, 3] = False
    assert np.array_equal(render_ref.outline(m), ring)
    full = np.ones((4, 5), bool)                       # outside the frame counts as unset
    border = full.copy()
    border[1:-1, 1:-1] = False
    assert np.array_equal(render_ref.outline(full), border)
    assert np.array_equal(render_ref.outline(np.ones((1, 1), bool)), np.ones((1, 1), bool))


def test_radius_zero_segments_cover_exactly_their_lattice_points():
    assert _seg_pixels(8, 9, 2, 3, 6, 3, 0) == {(x, 3) for x in range(2, 7)}
    assert _seg_pixels(8, 9, 4, 1, 4, 6, 0) == {(4, y) for y in range(1, 7)}
    assert _seg_pixels(8, 9, 1, 1, 5, 5, 0) == {(i, i) for i in range(1, 6)}
    assert _seg_pixels(8, 9, 0, 0, 4, 2, 0) == {(0, 0), (2, 1), (4, 2)}
    assert _seg_pixels(8, 9, 6, 3, 2, 3, 0) == {(x, 3) for x in range(2, 7)}         # direction does not matter


def test_point_segment_is_a_disc():
    got = _seg_pixels(11, 11, 5, 5, 5, 5, 2)
    assert got == {(x, y) for x in range(11) for y in range(11) if (x - 5) ** 2 + (y - 5) ** 2 <= 4}
    assert len(got) == 13
    assert _seg_pixels(11, 11, 5, 5, 5, 5, 0) == {(5, 5)}


def test_blend_rounding():
    # (c * a + o * (255 - a) + 127) // 255 in uint32
    for a, want in ((0, 100), (1, 100), (128, 150), (254, 200), (255, 200)):
        assert int(render_ref.blend(200, 100, a)) == want, a
    assert int(render_ref.blend(255, 0, 128)) == 128
    assert int(render_ref.blend(0, 255, 128)) == 127
    assert int(render_ref.blend(1, 0, 128)) == 1                       # 128 + 127 = 255 -> 1


def test_composite_order_fill_outline_segment():
    H, W = 6, 8
    m = np.zeros((1, H, W), bool)
    m[0, 1:5, 1:6] = True
    bg = np.full((H, W, 3), 10, np.uint8)
    lay, lb, sg, sb = _lists([(0, _lib.LAYER_FILL, (200, 0, 0, 255)), (0, _lib.LAYER_OUTLINE, (0, 200, 0, 255)),
                              (5, _lib.LAYER_FILL, (1, 2, 3, 255))],
                             [(0, 0, 0, 0, 0, (7, 8, 9), 0)])
    out = render_ref.composite(bg, m, lay, lb, sg, sb)[0]
    assert tuple(out[2, 2]) == (200, 0, 0)          # interior: fill only
    assert tuple(out[1, 1]) == (0, 200, 0)          # boundary: outline over the fill
    assert tuple(out[5, 7]) == (10, 10, 10)         # background; the out-of-pool layer draws nothing
    assert tuple(out[0, 0]) == (7, 8, 9)            # the segment is drawn last


def _clip():
    cfg = OptConfig()
    preds, _ = synth.make_video(5, 3, 6, cfg, kinds=[synth.KIND_TRANS, synth.KIND_ROT, synth.KIND_ROT])
    for t, p in enumerate(preds):
        p.scores = np.array([0.95, 0.9, 0.5 if t % 2 else 0.8])
    # rot track 1 is fitted, rot track 2 is not; frame 3's axis of track 1 misses the image
    preds[3].pred_rot_axis[1] = torch.tensor([0.6, 0.8, 100.0])
    planes = {"trans": [{"ids": {t: 0 for t in range(6)}, "has_rot": True}],
              "rot": [{"ids": {t: 1 for t in range(1, 6)}, "has_rot": True},
                      {"ids": {t: 2 for t in range(6)}, "has_rot": False}]}
    return cfg, preds, planes


def test_draw_lists_order_colours_threshold_and_axes():
    cfg, preds, planes = _clip()
    d = render.draw_lists(preds, planes, cfg, score_thresh=0.7)
    c0, c1, grey = (tuple(int(v) for v in c) for c in (render.PALETTE[0], render.PALETTE[1], render.GREY))
    assert d.n_reg == 6 + 5 and [len(p["ids"]) for p in d.fitted] == [6, 5]
    for t in range(6):
        L = d.layers[d.layer_begin[t]:d.layer_begin[t + 1]]
        want = [(t, _lib.LAYER_FILL, c0 + (128,))]
        if t >= 1:
            want.append((6 + t - 1, _lib.LAYER_FILL, c1 + (128,)))
        det = d.n_reg + 3 * t
        want += [(det, _lib.LAYER_OUTLINE, c0 + (255,))]
        if t >= 1:
            want.append((det + 1, _lib.LAYER_OUTLINE, c1 + (255,)))
        else:
            want.append((det + 1, _lib.LAYER_OUTLINE, grey + (255,)))       # box 1 of frame 0 is in no fitted track
        if t % 2 == 0:
            want.append((det + 2, _lib.LAYER_OUTLINE, grey + (255,)))       # unfitted track, score 0.8 >= 0.7
        assert [(int(x["mask"]), int(x["kind"]), tuple(int(v) for v in x["rgba"])) for x in L] == want, t
    # axes: the reference's border end-points, fallback rows skipped
    fallback = axis.angle_offset_to_axis_rows(np.array([[0.6, 0.8, 100.0]], np.float32),
                                              preds[3].pred_boxes.get_centers()[1:2].numpy())
    assert tuple(fallback[0]) == (0, 0, 1, 1)
    for t in range(6):
        S = d.segs[d.seg_begin[t]:d.seg_begin[t + 1]]
        ce = preds[t].pred_boxes.get_centers().numpy()
        tr = preds[t].pred_tran_axis[0].numpy()
        want = [(tuple(axis.angle_offset_to_axis_rows(np.array([[tr[0], tr[1], 0.0]], np.float32), ce[0:1])[0]), c0)]
        if t >= 1 and t != 3:
            row = axis.angle_offset_to_axis_rows(preds[t].pred_rot_axis[1:2].numpy(), ce[1:2])[0]
            want.append((tuple(row), c1))
        got = [((int(s["x0"]), int(s["y0"]), int(s["x1"]), int(s["y1"])), tuple(int(v) for v in s["rgb"])) for s in S]
        assert got == want, t
        assert all(int(s["radius"]) == 2 for s in S)


def test_draw_lists_threshold_hides_decayed_detections():
    cfg, preds, planes = _clip()
    d = render.draw_lists(preds, planes, cfg, score_thresh=0.99)
    assert not np.any(d.layers["kind"] == _lib.LAYER_OUTLINE)
    assert np.all(d.layers["kind"] == _lib.LAYER_FILL) and len(d.layers) == d.n_reg


def test_render_rejects_bad_arguments_before_any_device_work():
    bg = torch.zeros(4, 5, 3, dtype=torch.uint8)
    ok_seg = (0, 0, 3, 3, 1, (1, 2, 3), 0)
    bad = [
        dict(layers=[(0, _lib.LAYER_FILL, (1, 1, 1, 1))]),                  # mask outside an empty pool
        dict(segs=[(0, 0, (1 << 14) + 1, 0, 1, (1, 2, 3), 0)]),             # coordinate limit
        dict(segs=[(-(1 << 14) - 1, 0, 0, 0, 1, (1, 2, 3), 0)]),
        dict(segs=[(0, 0, 1, 1, 257, (1, 2, 3), 0)]),                       # radius limit
        dict(segs=[(0, 0, 1, 1, -1, (1, 2, 3), 0)]),
    ]
    for kw in bad:
        lay, lb, sg, sb = _lists(**kw)
        with pytest.raises(ValueError):
            engine.render(None, lay, lb, sg, sb, bg)
    lay, lb, sg, sb = _lists(segs=[ok_seg, ok_seg], T=2)
    with pytest.raises(ValueError):
        engine.render(None, lay, lb, sg, np.array([0, 2, 1]), bg)          # not monotone
    with pytest.raises(ValueError):
        engine.render(None, lay, lb, sg, np.array([0, 1, 1]), bg)          # does not end at the list length
    with pytest.raises(ValueError):
        engine.render(None, lay, lb, sg, np.array([1, 2, 2]), bg)          # does not start at 0
    with pytest.raises(ValueError):
        engine.render(None, lay, np.array([0, 0]), sg, sb, bg)             # frame counts disagree
    for b in (torch.zeros(4, 5, 4, dtype=torch.uint8), torch.zeros(4, 5, 3), torch.zeros(3, 4, 5, 3, dtype=torch.uint8),
              torch.zeros(0, 5, 3, dtype=torch.uint8), torch.zeros(4, 16385, 3, dtype=torch.uint8)):
        with pytest.raises(ValueError):
            engine.render(None, lay, lb, sg, sb, b)
    with pytest.raises(ValueError):
        engine.render(None, np.zeros(0, np.int32), lb, sg, sb, bg)          # not the a3d_layer_t dtype


def test_no_gpu_means_loud_failure():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lay, lb, sg, sb = _lists(segs=[(0, 0, 3, 3, 1, (1, 2, 3), 0)], T=2)
    with pytest.raises(_lib.A3DError):
        engine.render(None, lay, lb, sg, sb, torch.zeros(4, 5, 3, dtype=torch.uint8))
    cfg, preds, planes = _clip()
    with pytest.raises(_lib.A3DError):
        render.render_clip(preds, planes, cfg=cfg)
