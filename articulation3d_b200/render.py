"""The fitted articulation drawn into the clip's frames (row f5 of DESIGN.md §2): what the reference's
``tools/inference.py:253-278`` shows a user, rebuilt as a functional equivalent on the GPU rather than with
detectron2's ``Visualizer`` [3P-unverified: neither detectron2 nor matplotlib is available, so the picture is
not pinned to theirs].

Per frame, in this order:
  * every fitted track's registered mask of the frame (``plane['reg_masks']``), filled in the track's colour
    with alpha 128;
  * every detection whose (written-back) score is >= ``score_thresh``, outlined opaque: in its track's colour
    when its box belongs to a fitted track, grey otherwise (the write-back's score decay hides the detections
    the optimiser rejected);
  * every fitted track's articulation axis through the frame's box, radius 2, in the track's colour: the
    reference's integer border end-points (``axis.angle_offset_to_axis_rows``) of ``pred_rot_axis``, or of
    ``pred_tran_axis`` with a zero offset column for translation tracks.
Tracks are numbered as ``io.tracks_summary`` lists them (``trans``, then ``rot``); track k is drawn in
``PALETTE[k % len(PALETTE)]``.

``draw_lists`` builds the per-frame draw lists on the host; ``render_clip`` composites them on the device with
``engine.render`` straight from the packed registered masks (no dense mask is made); ``write_video`` renders
bounded chunks of frames and encodes one chunk on the host while the next renders.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, engine
from .axis import angle_offset_to_axis_rows
from .config import OptConfig

PALETTE = np.array([[31, 119, 180], [255, 127, 14], [44, 160, 44], [214, 39, 40], [148, 103, 189],
                    [140, 86, 75], [227, 119, 194], [188, 189, 34], [23, 190, 207], [255, 187, 120]], dtype=np.uint8)
GREY = np.array([128, 128, 128], dtype=np.uint8)
BACKGROUND_GREY = 160            # the flat image export.py textures with when there is no video
FILL_ALPHA = 128
AXIS_RADIUS = 2
_FALLBACK = (0, 0, 1, 1)         # angle_offset_to_axis's row for a line that misses the image
_INT64_MIN = -(2 ** 63)


@dataclass
class DrawLists:
    """Per-frame draw lists of a clip.  Pool order of the ``mask`` indices: the registered masks of every fitted
    track in track order (frames in ``plane['ids']`` order), then every detection mask in (frame, box) order."""
    layers: np.ndarray           # _lib.LAYER_DTYPE
    layer_begin: np.ndarray      # (T + 1,) int64
    segs: np.ndarray             # _lib.SEGMENT_DTYPE
    seg_begin: np.ndarray        # (T + 1,) int64
    fitted: list                 # plane dicts of the fitted tracks, in pool order
    n_reg: int                   # registered masks at the front of the pool


def _tracks(planes) -> list:
    """(is translation track, plane) in io.tracks_summary order."""
    return [(cat == "trans", plane) for cat in ("trans", "rot") for plane in planes[cat]]


def _has(p, name: str) -> bool:
    return p.has(name) if hasattr(p, "has") else hasattr(p, name)


def _flatten(per_frame, dtype):
    begin = np.zeros(len(per_frame) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in per_frame], out=begin[1:])
    arr = np.zeros(int(begin[-1]), dtype=dtype)
    for f, rows in enumerate(per_frame):
        for i, row in enumerate(rows):
            arr[begin[f] + i] = row
    return arr, begin


def draw_lists(opt_preds, planes, cfg: OptConfig | None = None, score_thresh: float = 0.7) -> DrawLists:
    """Layers and segments of every frame of a clip (host only; see the module docstring for what is drawn)."""
    cfg = cfg or OptConfig()
    H, W = cfg.height, cfg.width
    T = len(opt_preds)
    tracks = _tracks(planes)
    fitted = [(k, tr, pl) for k, (tr, pl) in enumerate(tracks) if pl.get("has_rot", False)]
    layers = [[] for _ in range(T)]
    segs = [[] for _ in range(T)]
    owner = {}
    base = 0
    for k, _, pl in fitted:
        col = tuple(int(c) for c in PALETTE[k % len(PALETTE)])
        for i, (f, b) in enumerate(pl["ids"].items()):
            layers[f].append((base + i, _lib.LAYER_FILL, col + (FILL_ALPHA,)))
            owner[(int(f), int(b))] = col
        base += len(pl["ids"])
    n_reg = base
    for f, p in enumerate(opt_preds):
        scores = np.asarray(p.scores, dtype=np.float64).reshape(-1)
        for b in np.flatnonzero(scores >= score_thresh):
            col = owner.get((f, int(b)), tuple(int(c) for c in GREY))
            layers[f].append((base + int(b), _lib.LAYER_OUTLINE, col + (255,)))
        base += len(scores)
    # axes: one row per (fitted track, frame), converted in one call
    ao, ce, where = [], [], []
    for k, trans, pl in fitted:
        for f, b in pl["ids"].items():
            p = opt_preds[f]
            if trans:
                t = np.asarray(p.pred_tran_axis[b], dtype=np.float32).reshape(2)
                ao.append([t[0], t[1], 0.0])
            else:
                ao.append(np.asarray(p.pred_rot_axis[b], dtype=np.float32).reshape(3))
            ce.append(np.asarray(p.pred_boxes.get_centers()[b], dtype=np.float32).reshape(2))
            where.append((f, k))
    if ao:
        rows = angle_offset_to_axis_rows(np.array(ao, np.float32), np.array(ce, np.float32), H=H, W=W)
        for (f, k), row in zip(where, rows):
            if tuple(row) == _FALLBACK or np.any(row == _INT64_MIN) or np.any(np.abs(row) > _lib.RENDER_MAX_COORD):
                continue                           # no line through the image, or one a3d_render cannot draw exactly
            col = tuple(int(c) for c in PALETTE[k % len(PALETTE)])
            segs[f].append(tuple(int(v) for v in row) + (AXIS_RADIUS, col, 0))
    lay, lb = _flatten(layers, _lib.LAYER_DTYPE)
    sg, sb = _flatten(segs, _lib.SEGMENT_DTYPE)
    return DrawLists(lay, lb, sg, sb, [pl for _, _, pl in fitted], n_reg)


def _device(device, planes) -> torch.device:
    if device is None:
        for _, pl in _tracks(planes):
            rm = pl.get("reg_masks")
            if pl.get("has_rot", False) and getattr(rm, "packed", None) is not None:
                device = rm.packed.device
                break
    device = torch.device(device if device is not None else "cuda")
    if device.type != "cuda" or not torch.cuda.is_available():
        raise _lib.A3DError("rendering needs a CUDA device (the hot path has no CPU fallback)")
    return device


def mask_pool(opt_preds, lists: DrawLists, cfg: OptConfig, device) -> engine.MaskPool:
    """The pool ``lists`` index: the fitted tracks' packed registered masks (``RegMasks.packed``, concatenated on
    the device), then the detection masks, packed from ``pred_masks`` or decoded from ``pred_rle`` on the device."""
    H, W = cfg.height, cfg.width
    parts = []
    for pl in lists.fitted:
        packed = getattr(pl.get("reg_masks"), "packed", None)
        if packed is None:
            raise TypeError("render needs the optimiser's packed registered masks (opt_utils.RegMasks)")
        parts.append(packed.to(device))
    n_det = sum(len(np.asarray(p.scores).reshape(-1)) for p in opt_preds)
    if n_det:
        if all(_has(p, "pred_masks") for p in opt_preds):
            builder = engine.PoolBuilder(n_det, H, W, device)
            for p in opt_preds:
                if len(p.pred_masks):
                    builder.append(torch.as_tensor(p.pred_masks).to(device))
            parts.append(builder.bits)
        else:
            rles = [r for p in opt_preds for r in p.pred_rle]
            parts.append(engine.rle_to_pool(rles, H, W, device).bits)
    if not parts:
        return None
    with torch.cuda.device(device):
        return engine.pool_from_bits(torch.cat(parts) if len(parts) > 1 else parts[0], H, W)


def _background(images, T: int, H: int, W: int, device):
    """(H, W, 3) uint8 on the device, or T frames (left where they are; moved to the device chunk by chunk)."""
    if images is None:
        return torch.full((H, W, 3), BACKGROUND_GREY, dtype=torch.uint8, device=device)
    img = torch.as_tensor(np.ascontiguousarray(images) if isinstance(images, np.ndarray) else images)
    if img.dtype != torch.uint8 or tuple(img.shape[-3:]) != (H, W, 3) or img.dim() not in (3, 4) \
            or (img.dim() == 4 and img.shape[0] != T):
        raise ValueError(f"images must be uint8 (H, W, 3) or ({T}, H, W, 3) with H, W = {H}, {W}")
    return img.to(device) if img.dim() == 3 else img


def _render_range(pool, lists: DrawLists, bg, a: int, b: int, device, out=None) -> torch.Tensor:
    lb, sb = lists.layer_begin, lists.seg_begin
    frame_bg = bg if bg.dim() == 3 else bg[a:b].to(device, non_blocking=True)
    return engine.render(pool, lists.layers[lb[a]:lb[b]], lb[a:b + 1] - lb[a], lists.segs[sb[a]:sb[b]],
                         sb[a:b + 1] - sb[a], frame_bg, out=out)


def render_clip(opt_preds, planes, images=None, cfg: OptConfig | None = None, device=None,
                score_thresh: float = 0.7) -> torch.Tensor:
    """(T, H, W, 3) uint8 RGB CUDA tensor of the clip drawn with the fitted result.  ``images``: None (flat grey),
    one (H, W, 3) uint8 image for every frame, or T frames."""
    cfg = cfg or OptConfig()
    device = _device(device, planes)
    lists = draw_lists(opt_preds, planes, cfg, score_thresh)
    pool = mask_pool(opt_preds, lists, cfg, device)
    bg = _background(images, len(opt_preds), cfg.height, cfg.width, device)
    with torch.cuda.device(device):
        return _render_range(pool, lists, bg, 0, len(opt_preds), device)


def write_video(path: str, opt_preds, planes, images=None, fps: float = 30, cfg: OptConfig | None = None,
                device=None, score_thresh: float = 0.7, chunk_bytes: int = 64 << 20) -> str:
    """``render_clip`` written as an mp4 (``cv2.VideoWriter``, ``mp4v``).  Frames are rendered in chunks of at most
    ``chunk_bytes`` of RGB; each chunk is copied into one of two pinned host buffers, and the host encodes a chunk
    while the device renders and copies the next."""
    import cv2
    cfg = cfg or OptConfig()
    H, W = cfg.height, cfg.width
    T = len(opt_preds)
    device = _device(device, planes)
    lists = draw_lists(opt_preds, planes, cfg, score_thresh)
    pool = mask_pool(opt_preds, lists, cfg, device)
    bg = _background(images, T, H, W, device)
    per = max(1, min(T, chunk_bytes // (H * W * 3)))
    writer = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (W, H))
    if not writer.isOpened():
        raise RuntimeError(f"cv2.VideoWriter cannot open {path}")

    def encode(host, done):
        done.synchronize()
        for frame in host.numpy():
            writer.write(cv2.cvtColor(frame, cv2.COLOR_RGB2BGR))

    try:
        with torch.cuda.device(device):
            pinned = [torch.empty((per, H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(min(2, -(-T // per)))]
            pending = None
            for c, a in enumerate(range(0, T, per)):
                b = min(T, a + per)
                frames = _render_range(pool, lists, bg, a, b, device)
                host = pinned[c % 2][:b - a]
                host.copy_(frames, non_blocking=True)
                done = torch.cuda.Event()
                done.record()
                if pending is not None:
                    encode(*pending)               # the previous chunk, while this one renders and copies
                pending = (host, done)
            if pending is not None:
                encode(*pending)
    finally:
        writer.release()
    return path
