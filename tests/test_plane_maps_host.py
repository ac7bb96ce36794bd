"""CPU tests of the plane maps: the numpy restatement of a3d_plane_maps on known answers, the layers
render.plane_lists builds, geometry.registered_planes against moved unprojected pixels, and engine.plane_maps'
argument checks (no GPU)."""
import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, geometry, render, synth
from tests import plane_maps_ref

KINV = OptConfig().K_inv()


def _layers(rows, T=1):
    lay = np.array(list(rows), dtype=_lib.PLANE_LAYER_DTYPE)
    lb = np.zeros(T + 1, np.int64)
    lb[1:] = len(lay)
    return lay, lb


def _row(mask, normal, offset, rgb):
    return (mask, normal, offset, rgb, 0)


def test_fronto_parallel_plane_gives_its_offset():
    H, W = 5, 7
    masks = np.ones((1, H, W), bool)
    lay, lb = _layers([_row(0, (0, 0, 1), 2.5, (1, 2, 3))])
    depth, rgb = plane_maps_ref.plane_maps(KINV, masks, lay, lb, (9, 9, 9))
    assert np.all(depth == np.float32(2.5)) and np.all(rgb == (1, 2, 3))
    # a general inverse with the same rays: z = d as well
    kinv = KINV * 2.0                              # rz = 2: depth = d / 2, z = depth * rz = d
    depth2, _ = plane_maps_ref.plane_maps(kinv, masks, lay, lb)
    assert np.all(depth2 == np.float32(2.5))


def test_nearer_of_two_overlapping_planes_wins_and_a_tie_goes_to_the_first():
    H, W = 4, 6
    masks = np.zeros((2, H, W), bool)
    masks[0, :, :4] = True
    masks[1, :, 2:] = True
    far, near = _row(0, (0, 0, 1), 3.0, (10, 0, 0)), _row(1, (0, 0, 1), 2.0, (0, 20, 0))
    for order in ((far, near), (near, far)):
        depth, rgb = plane_maps_ref.plane_maps(KINV, masks, *_layers(order), (5, 5, 5))
        assert np.all(depth[0, :, :2] == 3.0) and np.all(rgb[0, :, :2] == (10, 0, 0))
        assert np.all(depth[0, :, 2:] == 2.0) and np.all(rgb[0, :, 2:] == (0, 20, 0))
    a, b = _row(0, (0, 0, 1), 2.0, (1, 1, 1)), _row(1, (0, 0, 1), 2.0, (2, 2, 2))
    _, rgb = plane_maps_ref.plane_maps(KINV, masks, *_layers([a, b]))
    assert np.all(rgb[0, :, 2:4] == 1)
    _, rgb = plane_maps_ref.plane_maps(KINV, masks, *_layers([b, a]))
    assert np.all(rgb[0, :, 2:4] == 2)


def test_planes_behind_the_camera_edge_on_and_nan_cover_nothing():
    H, W = 3, 4
    masks = np.ones((1, H, W), bool)
    for normal, offset in (((0, 0, 1), -2.0), ((0, 0, 1), 0.0), ((1, 0, 0), 0.0), ((0, 0, 0), 1.0),
                           ((np.nan, 0, 1), 1.0), ((0, 0, 1), np.nan), ((0, 0, 1), np.inf)):
        depth, rgb = plane_maps_ref.plane_maps(KINV, masks, *_layers([_row(0, normal, offset, (7, 7, 7))]), (3, 4, 5))
        assert np.all(depth == 0) and np.all(rgb == (3, 4, 5)), (normal, offset)
    # edge-on: the plane x = 0 through the camera centre, seen along the column whose ray lies in it
    cfg = OptConfig()
    m = np.zeros((1, cfg.height, cfg.width), bool)
    m[0, 10, :] = True
    depth, _ = plane_maps_ref.plane_maps(KINV, m, *_layers([_row(0, (1, 0, 0), 0.0, (1, 1, 1))]))
    assert np.all(depth == 0)
    # out-of-pool masks cover nothing
    depth, _ = plane_maps_ref.plane_maps(KINV, masks, *_layers([_row(1, (0, 0, 1), 1.0, (1, 1, 1)),
                                                                 _row(-1, (0, 0, 1), 1.0, (1, 1, 1))]))
    assert np.all(depth == 0)


def test_normal_colours():
    c = render.normal_colours(np.array([[0, 0, -1], [0, 0, 1], [1, 0, 0], [-0.5, 0.25, np.nan]], np.float32))
    assert c.tolist() == [[128, 128, 255], [128, 128, 0], [0, 128, 128], [191, 96, 0]]


def _clip():
    cfg = OptConfig()
    preds, _ = synth.make_video(5, 3, 6, cfg, kinds=[synth.KIND_TRANS, synth.KIND_ROT, synth.KIND_ROT])
    for t, p in enumerate(preds):
        p.scores = np.array([0.95, 0.9, 0.5 if t % 2 else 0.8])
    rng = np.random.RandomState(0)

    def reg(n):
        r = rng.randn(n, 4).astype(np.float32)
        r[:, :3] /= np.linalg.norm(r[:, :3], axis=1, keepdims=True)
        return r
    planes = {"trans": [{"ids": {t: 0 for t in range(6)}, "has_rot": True, "fit": {"reg_plane": reg(6)}}],
              "rot": [{"ids": {t: 1 for t in range(1, 6)}, "has_rot": True, "fit": {"reg_plane": reg(5)}},
                      {"ids": {t: 2 for t in range(6)}, "has_rot": False}]}
    return cfg, preds, planes


def test_plane_lists_order_colours_fitted_boxes_and_threshold():
    cfg, preds, planes = _clip()
    d = render.plane_lists(preds, planes, cfg, score_thresh=0.7)
    r0, r1 = planes["trans"][0]["fit"]["reg_plane"], planes["rot"][0]["fit"]["reg_plane"]
    assert d.n_reg == 11 and [len(p["ids"]) for p in d.fitted] == [6, 5]
    lists = render.draw_lists(preds, planes, cfg, score_thresh=0.7)          # same pool
    assert lists.n_reg == d.n_reg and all(a is b for a, b in zip(lists.fitted, d.fitted))
    for t in range(6):
        L = d.layers[d.layer_begin[t]:d.layer_begin[t + 1]]
        want = [(t, r0[t])]
        if t >= 1:
            want.append((6 + t - 1, r1[t - 1]))
        det = d.n_reg + 3 * t
        if t == 0:
            want.append((det + 1, None))              # box 1 of frame 0 is in no fitted track
        if t % 2 == 0:
            want.append((det + 2, None))              # unfitted track, score 0.8 >= 0.7
        assert [int(x["mask"]) for x in L] == [m for m, _ in want], t
        for x, (m, reg) in zip(L, want):
            if reg is None:
                b = m - d.n_reg - 3 * t
                geo = synth_geometry(preds[t], b, cfg)
                reg = np.concatenate([geo.normal.numpy(), [geo.offset.item()]]).astype(np.float32)
            assert np.array_equal(x["normal"], reg[:3]) and x["offset"] == reg[3], (t, m)
            assert np.array_equal(x["rgb"], render.normal_colours(reg[None, :3])[0])
    d = render.plane_lists(preds, planes, cfg, score_thresh=0.99)
    assert len(d.layers) == d.n_reg


def synth_geometry(p, b, cfg):
    return geometry.source_geometry(p, b, cfg, translation=False)


def _moved_residual(rows, cand, mode, pivot, pts, reg, transpose=False):
    """max |n' . p' - d'| / (1 + |p'| + |d'|) over the points p moved by each candidate in float64."""
    worst = 0.0
    for i, c in enumerate(cand):
        R = rows[c, :9].reshape(3, 3).astype(np.float64)
        if transpose:
            R = R.T
        if mode == _lib.MODE_SEQ:
            a = pivot.astype(np.float64)
            q = (pts - a) @ R + a
        else:
            q = pts @ R + rows[c, 9:].astype(np.float64)
        n, dd = reg[i, :3].astype(np.float64), np.float64(reg[i, 3])
        err = np.abs(q @ n - dd) / (1 + np.abs(q).sum(1) + abs(dd))
        worst = max(worst, float(err.max()))
    return worst


@pytest.mark.parametrize("mode", [_lib.MODE_COMPOSED, _lib.MODE_TRANSLATE, _lib.MODE_SEQ],
                         ids=["composed", "translate", "seq"])
def test_registered_planes_contain_the_moved_pixels(mode):
    cfg = OptConfig()
    preds, _ = synth.make_video(8, 2, 4, cfg, kinds=[synth.KIND_ROT, synth.KIND_TRANS])
    b = 1 if mode == _lib.MODE_TRANSLATE else 0
    geo = geometry.source_geometry(preds[2], b, cfg, translation=mode == _lib.MODE_TRANSLATE)
    ys, xs = np.nonzero(preds[2].pred_masks[b].numpy() > 0.5)
    sel = np.linspace(0, len(xs) - 1, 200).astype(int)
    pts = geometry.unproject_points(np.stack([xs[sel], ys[sel]], 1), geo.normal, geo.offset, cfg)
    if mode == _lib.MODE_TRANSLATE:
        rows = geometry.xforms_translate(cfg.trans_grid, geo.dir_vec)
    elif mode == _lib.MODE_SEQ:
        rows = geometry.xforms_seq_from_dirs(cfg.legacy_grid, geo.dir_vec)
    else:
        rows = geometry.xforms_composed(geometry.rotation_matrices(cfg.rot_final_grid, geo.dir_vec), geo.pivot)
    cand = np.arange(len(rows))[::-1]
    reg = geometry.registered_planes(geo.normal, geo.offset, rows, mode, geo.pivot, cand)
    assert reg.dtype == np.float32 and reg.shape == (len(rows), 4)
    assert _moved_residual(rows, cand, mode, geo.pivot, pts, reg) < 1e-6
    if mode != _lib.MODE_TRANSLATE:
        # the test would catch R and R^T mixed up
        assert _moved_residual(rows, cand, mode, geo.pivot, pts, reg, transpose=True) > 1e-3
        want = geometry.transform_normals(geo.normal, rows[:, :9].reshape(-1, 3, 3)).numpy()[cand]
        assert np.array_equal(reg[:, :3], want)
    else:
        assert np.array_equal(reg[:, :3], np.broadcast_to(geo.normal.numpy(), (len(rows), 3)))


def test_plane_maps_rejects_bad_arguments_before_any_device_work():
    cfg = OptConfig.scaled(40, 30)
    lay, lb = _layers([], T=2)
    with pytest.raises(ValueError):
        engine.plane_maps(None, *_layers([_row(0, (0, 0, 1), 1.0, (1, 1, 1))]), cfg)     # mask outside an empty pool
    with pytest.raises(ValueError):
        engine.plane_maps(None, np.zeros(0, _lib.LAYER_DTYPE), lb, cfg)                  # not a3d_plane_layer_t
    for begin in (np.array([0, 1, 0]), np.array([1, 0, 0]), np.array([0, 0, 1]), np.array([0.0, 0.0]), np.zeros(0)):
        with pytest.raises(ValueError):
            engine.plane_maps(None, lay, begin, cfg)
    for bg in ((0, 0), (0, 0, 256), (-1, 0, 0), (0.5, 0, 0)):
        with pytest.raises(ValueError):
            engine.plane_maps(None, lay, lb, cfg, bg)
    for c in (OptConfig.scaled(16386, 30), OptConfig(height=0, width=640)):
        with pytest.raises(ValueError):
            engine.plane_maps(None, lay, lb, c)
    for kw in (dict(depth_out=torch.zeros(2, 30, 40, dtype=torch.float64)), dict(depth_out=torch.zeros(1, 30, 40)),
               dict(depth_out=torch.zeros(2, 40, 30).transpose(1, 2)),
               dict(rgb_out=torch.zeros(2, 30, 40, 3)), dict(rgb_out=torch.zeros(2, 30, 40, 4, dtype=torch.uint8))):
        with pytest.raises(ValueError):
            engine.plane_maps(None, lay, lb, cfg, **kw)


def test_no_gpu_means_loud_failure():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = OptConfig.scaled(40, 30)
    with pytest.raises(_lib.A3DError):
        engine.plane_maps(None, *_layers([], T=2), cfg)
    cfg, preds, planes = _clip()
    with pytest.raises(_lib.A3DError):
        render.plane_maps(preds, planes, cfg=cfg)
