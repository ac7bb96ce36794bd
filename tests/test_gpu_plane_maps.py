"""GPU tests of the plane maps: a3d_plane_maps bit for bit against the numpy restatement (tests/plane_maps_ref.py) at
frame sizes from 1x1 to 2048x2048 with sparse and general intrinsics, render.plane_maps after the optimiser against
the synthetic scene's true depth, and the tools' --save-depth."""
import filecmp
import os
import random

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, opt_utils, render, synth
from tests import plane_maps_ref
from tests.test_gpu_render import _masks, _video_frames      # pools that touch every border; mp4 read-back

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SHAPES = [(1, 1), (31, 33), (480, 640), (768, 1024), (2048, 2048)]


def _cfg(H, W, kind):
    cfg = OptConfig.scaled(W, H)
    if kind == "general":                  # skew, non-square pixels and a slightly rotated camera: rz != 1
        K = np.array([[cfg.focal_length * 1.05, 12.0, cfg.cx + 7.0], [0.0, cfg.focal_length * 0.93, cfg.cy - 5.0],
                      [0.0, 0.0, 1.0]])
        c, s = np.cos(0.05), np.sin(0.05)
        kinv = np.array([[1.0, 0.0, 0.0], [0.0, c, -s], [0.0, s, c]]) @ np.linalg.inv(K)
        cfg.K_inv = lambda: kinv                                       # what engine.camera_struct reads
    return cfg


def _layers(T, n_masks, rng, per_frame=6):
    """Random planes in front of the camera, with ties, planes behind it, NaN and zero normals."""
    rows, lb = [], [0]
    for f in range(T):
        k = per_frame if f % 3 != 2 else 0                            # every third frame has no layers
        for i in range(k):
            n = rng.randn(3)
            n[2] = abs(n[2]) + 0.3
            n /= np.linalg.norm(n)
            off = rng.uniform(0.5, 5.0)
            r = rng.rand()
            if r < 0.08:
                off = -off                                             # behind the camera
            elif r < 0.12:
                n = np.array([np.nan, 0.0, 1.0])
            elif r < 0.15:
                n = np.zeros(3)
            rows.append((rng.randint(0, n_masks), n, off, tuple(rng.randint(0, 256, 3)), 0))
            if i == 0:                                                 # a tie: same plane, another colour
                rows.append((rng.randint(0, n_masks), n, off, tuple(rng.randint(0, 256, 3)), 0))
        lb.append(len(rows))
    return np.array(rows, dtype=_lib.PLANE_LAYER_DTYPE), np.array(lb, np.int64)


def _pool(masks):
    return engine.pack_masks(torch.from_numpy(masks.astype(np.uint8)).to(DEV))


def _raw(cfg, pool, bbox, lay, lb, bg, depth, rgb):
    """a3d_plane_maps through the C ABI (bbox may be None)."""
    lib = _lib.load()
    d_lay = torch.from_numpy(np.ascontiguousarray(lay).view(np.uint8).copy()).to(DEV) if len(lay) else None
    d_lb = torch.from_numpy(lb.astype(np.int64)).to(DEV)
    cam = engine.camera_struct(cfg)
    import ctypes
    rc = lib.a3d_plane_maps(ctypes.byref(cam), len(lb) - 1, pool.bits.data_ptr(), bbox, len(pool),
                            d_lay.data_ptr() if d_lay is not None else None, d_lb.data_ptr(),
                            (ctypes.c_uint8 * 3)(*bg), depth.data_ptr() if depth is not None else None,
                            rgb.data_ptr() if rgb is not None else None, torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.a3d_last_error_string()
    torch.cuda.synchronize()


def _check(cfg, masks, lay, lb, bg=(17, 34, 51)):
    pool = _pool(masks)
    depth, rgb = engine.plane_maps(pool, lay, lb, cfg, bg)
    want_d, want_c = plane_maps_ref.plane_maps(cfg.K_inv(), masks, lay, lb, bg)
    got_d = depth.view(torch.int32).cpu().numpy()
    bad = np.argwhere(got_d != want_d.view(np.int32))
    assert len(bad) == 0, f"{len(bad)} depths differ, first at {bad[:5].tolist()}"
    assert np.array_equal(rgb.cpu().numpy(), want_c)
    d2, c2 = torch.full_like(depth, 7.0), torch.full_like(rgb, 7)      # without boxes: no culling, same output
    _raw(cfg, pool, None, lay, lb, bg, d2, c2)
    assert np.array_equal(d2.view(torch.int32).cpu().numpy(), want_d.view(np.int32))
    assert np.array_equal(c2.cpu().numpy(), want_c)
    return want_d, want_c


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("kind", ["sparse", "general"])
def test_plane_maps_equal_restatement(shape, kind):
    H, W = shape
    cfg = _cfg(H, W, kind)
    rng = np.random.RandomState(H * 31 + W + len(kind))
    T = 2 if H * W > 10 ** 6 else 5
    masks = _masks(6, H, W, rng)
    lay, lb = _layers(T, len(masks), rng)
    want_d, _ = _check(cfg, masks, lay, lb)
    if H * W > 100:
        assert np.count_nonzero(want_d) > 0


def test_more_layers_than_one_culling_batch_and_ties_across_batches():
    H, W = 37, 70
    cfg = _cfg(H, W, "sparse")
    rng = np.random.RandomState(3)
    masks = _masks(40, H, W, rng)
    lay, lb = _layers(4, len(masks), rng, per_frame=300)
    # frame 0: the same plane at the ends of two different batches; the first must win
    lay[0] = (0, (0.0, 0.0, 1.0), 1.0, (1, 2, 3), 0)
    lay[lb[1] - 1] = (0, (0.0, 0.0, 1.0), 1.0, (9, 9, 9), 0)
    assert lb[1] - lb[0] > 256                                      # the kernel culls 256 layers per batch
    _, want_c = _check(cfg, masks, lay, lb)
    assert np.any(np.all(want_c[0] == (1, 2, 3), axis=-1))
    assert not np.any(np.all(want_c[0] == (9, 9, 9), axis=-1))


def test_out_of_range_masks_cover_nothing_and_only_the_outputs_are_written():
    H, W, T = 13, 37, 3
    cfg = _cfg(H, W, "sparse")
    rng = np.random.RandomState(4)
    masks = _masks(3, H, W, rng)
    pool = _pool(masks)
    front = (0.0, 0.0, 1.0)
    lay = np.array([(-1, front, 1.0, (9, 9, 9), 0), (3, front, 1.0, (9, 9, 9), 0), (1 << 30, front, 1.0, (9, 9, 9), 0),
                    (1, front, 2.0, (200, 100, 0), 0)], dtype=_lib.PLANE_LAYER_DTYPE)
    lb = np.array([0, 4, 4, 4])
    want_d, want_c = plane_maps_ref.plane_maps(cfg.K_inv(), masks, lay, lb, (5, 6, 7))
    nd, nc = T * H * W, T * H * W * 3
    dbuf = torch.full((nd + 16,), -3.0, device=DEV)
    cbuf = torch.full((nc + 64,), 0xAB, dtype=torch.uint8, device=DEV)
    for bbox in (pool.bbox.data_ptr(), None):
        _raw(cfg, pool, bbox, lay, lb, (5, 6, 7), dbuf[8:8 + nd], cbuf[32:32 + nc])
        d, c = dbuf.cpu().numpy(), cbuf.cpu().numpy()
        assert np.all(d[:8] == -3.0) and np.all(d[8 + nd:] == -3.0)
        assert np.all(c[:32] == 0xAB) and np.all(c[32 + nc:] == 0xAB)
        assert np.array_equal(d[8:8 + nd].reshape(T, H, W).view(np.int32), want_d.view(np.int32))
        assert np.array_equal(c[32:32 + nc].reshape(T, H, W, 3), want_c)
    assert np.all(want_d[1:] == 0) and np.all(want_c[1:] == (5, 6, 7))
    # either output alone
    d1 = torch.zeros(T, H, W, device=DEV)
    _raw(cfg, pool, pool.bbox.data_ptr(), lay, lb, (5, 6, 7), d1, None)
    assert np.array_equal(d1.cpu().numpy().view(np.int32), want_d.view(np.int32))
    c1 = torch.zeros(T, H, W, 3, dtype=torch.uint8, device=DEV)
    _raw(cfg, pool, pool.bbox.data_ptr(), lay, lb, (5, 6, 7), None, c1)
    assert np.array_equal(c1.cpu().numpy(), want_c)


def _optimised(cfg, seed=11, T=30):
    preds, scene = synth.make_video(seed, 4, T, cfg, kinds=[synth.KIND_ROT, synth.KIND_TRANS, synth.KIND_ROT,
                                                            synth.KIND_STATIC])
    random.seed(seed)
    planes = opt_utils.track_planes(preds, cfg)
    out = opt_utils.optimize_planes(preds, planes, '3dc', cfg=cfg, device=DEV)
    return out, planes, scene


def test_plane_maps_after_optimize_against_the_true_depth():
    cfg = OptConfig()
    opt, planes, scene = _optimised(cfg)
    fitted = [pl for cat in ("trans", "rot") for pl in planes[cat] if pl["has_rot"]]
    assert len(fitted) >= 2
    depth, rgb = render.plane_maps(opt, planes, cfg=cfg, device=DEV)
    assert depth.is_cuda and depth.shape == (30, 480, 640) and rgb.shape == (30, 480, 640, 3)
    depth, rgb = depth.cpu().numpy(), rgb.cpu().numpy()
    # bit for bit the restatement of the same lists
    lists = render.plane_lists(opt, planes, cfg)
    masks = [pl["reg_masks"][f].numpy() > 0.5 for pl in lists.fitted for f in pl["ids"]]
    masks += [m.numpy() > 0.5 for p in opt for m in p.pred_masks]
    want_d, want_c = plane_maps_ref.plane_maps(cfg.K_inv(), np.stack(masks), lists.layers, lists.layer_begin)
    assert np.array_equal(depth.view(np.int32), want_d.view(np.int32)) and np.array_equal(rgb, want_c)
    # against the scene: the true plane c.X = |c|^2 of each track, seen through the optimiser's camera
    ray = plane_maps_ref.rays(cfg.K_inv(), cfg.height, cfg.width)
    true_planes = synth.scene_planes(scene).numpy()
    errs = []
    for pl in lists.fitted:
        reg = pl["fit"]["reg_plane"]
        cols = render.normal_colours(reg[:, :3])
        for i, (f, b) in enumerate(pl["ids"].items()):
            k = int(b)                                   # no dropped detections: box b is scene track b
            true_mask = synth.render_track_masks(scene, k, cfg)[f].numpy()
            c = true_planes[k, f]
            z_true = (c @ c) / (c[0] * ray[0] + c[1] * ray[1] + c[2] * ray[2]) * ray[2]
            z_reg = plane_maps_ref.plane_z(ray, reg[i, :3], reg[i, 3])
            wins = (pl["reg_masks"][f].numpy() > 0.5) & (depth[f] == z_reg) & (z_reg > 0)
            assert np.all(rgb[f][wins] == cols[i]), (f, k)
            both = wins & true_mask
            if both.any():
                errs.append(np.abs(depth[f][both] - z_true[both]) / z_true[both])
    err = float(np.median(np.concatenate(errs)))
    print(f"median relative depth error of the fitted planes: {err:.4f} over {sum(map(len, errs))} pixels")
    assert err < 0.10


def _pngs(d):
    import cv2
    names = sorted(os.listdir(d))
    imgs = [cv2.imread(os.path.join(d, n), cv2.IMREAD_UNCHANGED) for n in names]
    return names, imgs


def _same_files(a, b):
    """Every file of directory a exists in b with the same bytes."""
    for name in os.listdir(a):
        assert filecmp.cmp(os.path.join(a, name), os.path.join(b, name), shallow=False), name


def _check_depth_outputs(out, vid, T, H=480, W=640):
    names, imgs = _pngs(os.path.join(out, f"{vid}_depth"))
    assert names == [f"{k:05d}.png" for k in range(T)]
    assert all(im.dtype == np.uint16 and im.shape == (H, W) for im in imgs)
    assert any(np.count_nonzero(im) for im in imgs)
    assert _video_frames(os.path.join(out, f"{vid}_normals.mp4")) == (T, (H, W, 3))


def test_write_plane_maps_chunks_match_plane_maps(tmp_path):
    import cv2
    cfg = OptConfig()
    opt, planes, _ = _optimised(cfg, seed=12, T=20)
    depth, _ = render.plane_maps(opt, planes, cfg=cfg, device=DEV)
    render.write_plane_maps(str(tmp_path), "v", opt, planes, cfg=cfg, device=DEV, chunk_bytes=7 * 640 * 480 * 5)
    _check_depth_outputs(str(tmp_path), "v", 20)
    mm = (depth * 1000.0).round().clamp(0, 65535).to(torch.int32).cpu().numpy()
    for k in range(20):
        assert np.array_equal(cv2.imread(str(tmp_path / "v_depth" / f"{k:05d}.png"), cv2.IMREAD_UNCHANGED), mm[k])


def test_inference_save_depth(tmp_path):
    from articulation3d_b200.tools import inference
    a, b = tmp_path / "a", tmp_path / "b"
    inference.main(["--output", str(a), "--frames", "20", "--device", DEV])
    inference.main(["--output", str(b), "--frames", "20", "--save-depth", "--device", DEV])
    _check_depth_outputs(str(b), "synthetic00_0_0", 20)
    assert set(os.listdir(b)) == set(os.listdir(a)) | {"synthetic00_0_0_depth", "synthetic00_0_0_normals.mp4"}
    _same_files(a, b)


def test_opt_arti_save_depth(tmp_path):
    from articulation3d_b200.tools import opt_arti
    inp, a, b = str(tmp_path / "in.pth"), tmp_path / "a", tmp_path / "b"
    opt_arti.main(["--input", inp, "--output", str(a), "--synthetic", "2", "--frames", "12", "--tracks", "3"])
    opt_arti.main(["--input", inp, "--output", str(b), "--save-depth"])
    new = set()
    for v in range(2):
        vid = f"synthetic{v:02d}_0_0"
        _check_depth_outputs(str(b), vid, 12)
        new |= {f"{vid}_depth", f"{vid}_normals.mp4"}
    assert set(os.listdir(b)) == set(os.listdir(a)) | new
    _same_files(a, b)
