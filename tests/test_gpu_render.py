"""GPU tests of the clip renderer: a3d_render byte for byte against the numpy restatement (tests/render_ref.py) at
frame sizes from 1x1 to 2048x2048, render.render_clip after the optimiser, and the tools' --save-video."""
import os
import random

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, io, opt_utils, render, rle, synth
from tests import render_ref

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
SHAPES = [(1, 1), (1, 1000), (7, 33), (9, 63), (31, 65), (480, 640), (768, 1024), (2048, 2048)]


def _masks(n, H, W, rng):
    """Random pool that touches every border: full, border lines, boxes, noise, empty."""
    m = np.zeros((n, H, W), bool)
    m[0] = True
    m[1, 0, :] = m[1, H - 1, :] = m[1, :, 0] = m[1, :, W - 1] = True
    for i in range(2, n - 1):
        if i % 2:
            m[i] = rng.rand(H, W) < 0.4
        else:
            y0, x0 = rng.randint(0, H), rng.randint(0, W)
            m[i, y0:y0 + rng.randint(1, H + 1), x0:x0 + rng.randint(1, W + 1)] = True
    return m                                           # the last mask stays empty


def _lists(T, n_masks, H, W, rng, n_layers=5, n_segs=3):
    lay, seg = [], []
    lb, sb = [0], [0]
    for f in range(T):
        k = n_layers if f % 3 != 2 else 0              # every third frame has no layers
        for _ in range(k):
            a = int(rng.choice([0, 1, 128, 200, 254, 255]))
            lay.append((rng.randint(0, n_masks), rng.randint(0, 2), tuple(rng.randint(0, 256, 3)) + (a,)))
        s = n_segs if f % 4 != 3 else 0
        for _ in range(s):
            x0, x1 = rng.randint(-20, W + 20, 2)
            y0, y1 = rng.randint(-20, H + 20, 2)
            if rng.rand() < 0.2:
                x1, y1 = x0, y0                        # degenerate: a disc
            seg.append((x0, y0, x1, y1, rng.randint(0, 6), tuple(rng.randint(0, 256, 3)), 0))
        lb.append(len(lay))
        sb.append(len(seg))
    return (np.array(lay, dtype=_lib.LAYER_DTYPE), np.array(lb, np.int64),
            np.array(seg, dtype=_lib.SEGMENT_DTYPE), np.array(sb, np.int64))


def _pool(masks):
    return engine.pack_masks(torch.from_numpy(masks.astype(np.uint8)).to(DEV))


def _raw(bg, pool, bbox, n_masks, lay, lb, sg, sb, out):
    """a3d_render through the C ABI (bbox may be None)."""
    lib = _lib.load()
    dev = [torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).copy()).to(DEV) if len(a) else None
           for a in (lay, lb, sg, sb)]
    H, W = bg.shape[-3], bg.shape[-2]
    stride = H * W * 3 if bg.dim() == 4 else 0
    rc = lib.a3d_render(bg.data_ptr(), stride, len(lb) - 1, H, W, pool.bits.data_ptr() if pool is not None else None,
                        bbox, n_masks, *(d.data_ptr() if d is not None else None for d in dev), out.data_ptr(),
                        torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.a3d_last_error_string()
    torch.cuda.synchronize()


def _check(bg_np, masks, lay, lb, sg, sb):
    pool = _pool(masks) if len(masks) else None
    bg = torch.from_numpy(bg_np).to(DEV)
    got = engine.render(pool, lay, lb, sg, sb, bg).cpu().numpy()
    want = render_ref.composite(bg_np, masks, lay, lb, sg, sb)
    assert got.shape == want.shape
    bad = np.argwhere(got != want)
    assert len(bad) == 0, f"{len(bad)} bytes differ, first at {bad[:5].tolist()}"
    if pool is not None:                               # without boxes: no culling, same bytes
        out = torch.empty_like(torch.from_numpy(got)).to(DEV)
        _raw(bg, pool, None, len(pool), lay, lb, sg, sb, out)
        assert np.array_equal(out.cpu().numpy(), want)
    return got


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
@pytest.mark.parametrize("per_frame", [False, True], ids=["shared_bg", "frame_bg"])
def test_render_equals_restatement(shape, per_frame):
    H, W = shape
    rng = np.random.RandomState(H * 31 + W + per_frame)
    T = 2 if H * W > 10 ** 6 else 7
    masks = _masks(6, H, W, rng)
    lists = _lists(T, len(masks), H, W, rng)
    bg = rng.randint(0, 256, (T, H, W, 3) if per_frame else (H, W, 3)).astype(np.uint8)
    _check(bg, masks, *lists)


def test_fill_and_outline_order_matters():
    H, W = 40, 70
    rng = np.random.RandomState(1)
    masks = _masks(4, H, W, rng)
    fill, outl = (2, _lib.LAYER_FILL, (250, 10, 10, 128)), (2, _lib.LAYER_OUTLINE, (10, 250, 10, 200))
    lay = np.array([fill, outl, outl, fill], dtype=_lib.LAYER_DTYPE)
    sg = np.zeros(0, _lib.SEGMENT_DTYPE)
    bg = np.full((H, W, 3), 90, np.uint8)
    got = _check(bg, masks, lay, np.array([0, 2, 4]), sg, np.zeros(3, np.int64))
    assert not np.array_equal(got[0], got[1])


def test_frames_without_layers_or_segments_are_the_background():
    H, W = 17, 45
    rng = np.random.RandomState(2)
    bg = rng.randint(0, 256, (3, H, W, 3)).astype(np.uint8)
    lay, sg = np.zeros(0, _lib.LAYER_DTYPE), np.zeros(0, _lib.SEGMENT_DTYPE)
    got = _check(bg, np.zeros((0, H, W), bool), lay, np.zeros(4, np.int64), sg, np.zeros(4, np.int64))
    assert np.array_equal(got, bg)


def test_segments_degenerate_off_image_and_at_the_limits():
    H, W = 480, 640
    L, R = 1 << 14, 256
    segs = [(-L, -L, L, L, R, (1, 2, 3), 0), (L, -L, -L, L, 2, (4, 5, 6), 0), (-L, 100, L, 101, 0, (7, 8, 9), 0),
            (320, 240, 320, 240, R, (10, 11, 12), 0), (-300, -300, -300, -300, R, (13, 14, 15), 0),   # disc off image
            (W + 255, 10, W + 255, 400, R, (16, 17, 18), 0), (W + 257, 10, W + 257, 400, R, (19, 20, 21), 0),
            (5, 5, 5, 5, 0, (22, 23, 24), 0), (0, 0, W - 1, H - 1, 0, (25, 26, 27), 0),
            (-L, -L, -L, L, R, (28, 29, 30), 0), (3, -L, 3, L, 0, (31, 32, 33), 0)]
    sg = np.array(segs, dtype=_lib.SEGMENT_DTYPE)
    bg = np.full((H, W, 3), 50, np.uint8)
    for order in (sg, sg[::-1].copy()):
        _check(bg, np.zeros((0, H, W), bool), np.zeros(0, _lib.LAYER_DTYPE), np.zeros(2, np.int64), order,
               np.array([0, len(sg)]))


def test_300_frames_of_32_layers():
    H, W = 48, 80
    rng = np.random.RandomState(3)
    masks = _masks(40, H, W, rng)
    lists = _lists(300, len(masks), H, W, rng, n_layers=32, n_segs=4)
    _check(np.full((H, W, 3), 160, np.uint8), masks, *lists)


def test_out_of_range_masks_draw_nothing_and_write_only_out():
    H, W, T = 13, 37, 3
    rng = np.random.RandomState(4)
    masks = _masks(3, H, W, rng)
    pool = _pool(masks)
    lay = np.array([(-1, 0, (9, 9, 9, 255)), (3, 1, (9, 9, 9, 255)), (1 << 30, 0, (9, 9, 9, 255)),
                    (1, 0, (200, 100, 0, 255))], dtype=_lib.LAYER_DTYPE)
    lb = np.array([0, 4, 4, 4])
    sg, sb = np.zeros(0, _lib.SEGMENT_DTYPE), np.zeros(T + 1, np.int64)
    bg_np = rng.randint(0, 256, (H, W, 3)).astype(np.uint8)
    bg = torch.from_numpy(bg_np).to(DEV)
    n = T * H * W * 3
    buf = torch.full((n + 64,), 0xAB, dtype=torch.uint8, device=DEV)
    out = buf[32:32 + n]                                     # 32 guard bytes on either side
    for bbox in (pool.bbox.data_ptr(), None):
        _raw(bg, pool, bbox, len(pool), lay, lb, sg, sb, out)
        b = buf.cpu().numpy()
        assert np.all(b[:32] == 0xAB) and np.all(b[32 + n:] == 0xAB)
        want = render_ref.composite(bg_np, masks, lay, lb, sg, sb)
        assert np.array_equal(b[32:32 + n].reshape(T, H, W, 3), want)
    assert np.all(want[1:] == bg_np)


def _optimised(cfg, masks="dense", seed=11):
    preds, _ = synth.make_video(seed, 4, 30, cfg, kinds=[synth.KIND_ROT, synth.KIND_TRANS, synth.KIND_ROT,
                                                         synth.KIND_STATIC])
    if masks == "rle":
        recs = io.preds_to_records(preds, device=DEV)
        preds = io.records_to_preds(recs, conf_threshold=0.7, masks="rle")
    random.seed(seed)
    planes = opt_utils.track_planes(preds, cfg)
    out = opt_utils.optimize_planes(preds, planes, '3dc', cfg=cfg, device=DEV)
    return out, planes


def _expected(opt, planes, cfg, images):
    lists = render.draw_lists(opt, planes, cfg)
    masks = [pl["reg_masks"][f].numpy() > 0.5 for pl in lists.fitted for f in pl["ids"]]
    for p in opt:
        if p.has("pred_masks"):
            masks += [m.numpy() > 0.5 for m in p.pred_masks]
        else:
            masks += [rle.decode(r) != 0 for r in p.pred_rle]
    bg = np.full((cfg.height, cfg.width, 3), 160, np.uint8) if images is None else images
    return render_ref.composite(bg, np.stack(masks), lists.layers, lists.layer_begin, lists.segs, lists.seg_begin)


@pytest.mark.parametrize("case", ["640x480", "1024x768", "dense_images", "rle"])
def test_render_clip_after_optimize(case):
    cfg = OptConfig.scaled(1024, 768) if case == "1024x768" else OptConfig()
    opt, planes = _optimised(cfg, masks="rle" if case == "rle" else "dense")
    assert any(pl["has_rot"] for cat in ("trans", "rot") for pl in planes[cat])
    images = None
    if case == "dense_images":
        images = np.random.RandomState(5).randint(0, 256, (30, cfg.height, cfg.width, 3)).astype(np.uint8)
    got = render.render_clip(opt, planes, images=images, cfg=cfg, device=DEV)
    assert got.is_cuda and got.shape == (30, cfg.height, cfg.width, 3) and got.dtype == torch.uint8
    assert np.array_equal(got.cpu().numpy(), _expected(opt, planes, cfg, images))


def _video_frames(path):
    import cv2
    cap = cv2.VideoCapture(path)
    assert cap.isOpened(), path
    n, shape = 0, None
    while True:
        ok, frame = cap.read()
        if not ok:
            break
        n, shape = n + 1, frame.shape
    cap.release()
    return n, shape


def test_write_video_chunks_match_render_clip(tmp_path):
    cfg = OptConfig()
    opt, planes = _optimised(cfg)
    path = render.write_video(str(tmp_path / "v.mp4"), opt, planes, cfg=cfg, device=DEV, chunk_bytes=7 * 640 * 480 * 3)
    assert _video_frames(path) == (30, (480, 640, 3))


def test_inference_save_video(tmp_path):
    from articulation3d_b200.tools import inference
    inference.main(["--output", str(tmp_path), "--frames", "20", "--save-video", "--device", DEV])
    assert _video_frames(str(tmp_path / "synthetic00_0_0.mp4")) == (20, (480, 640, 3))


def test_opt_arti_save_video_with_image_root(tmp_path):
    import cv2
    from articulation3d_b200.tools import opt_arti
    root = tmp_path / "images"
    root.mkdir()
    rng = np.random.RandomState(6)
    for v in range(2):
        for t in range(10):
            cv2.imwrite(str(root / f"synthetic{v:02d}_0_0_{t}.png"), rng.randint(0, 256, (480, 640, 3)).astype(np.uint8))
    inp, out = str(tmp_path / "in.pth"), tmp_path / "out"
    opt_arti.main(["--input", inp, "--output", str(out), "--synthetic", "2", "--frames", "10", "--tracks", "3",
                   "--save-video", "--image-root", str(root)])
    for v in range(2):
        assert _video_frames(str(out / f"synthetic{v:02d}_0_0.mp4")) == (10, (480, 640, 3))
    # a missing or wrongly sized image stops the tool before it writes anything
    os.remove(root / "synthetic01_0_0_4.png")
    with pytest.raises(SystemExit, match="cannot read"):
        opt_arti.main(["--input", inp, "--output", str(tmp_path / "o2"), "--save-video", "--image-root", str(root)])
    cv2.imwrite(str(root / "synthetic01_0_0_4.png"), np.zeros((240, 320, 3), np.uint8))
    with pytest.raises(SystemExit, match="320x240"):
        opt_arti.main(["--input", inp, "--output", str(tmp_path / "o2"), "--save-video", "--image-root", str(root)])
    assert not (tmp_path / "o2").exists()
