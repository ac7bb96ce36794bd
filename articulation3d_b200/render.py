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

The 3-D half of the result (row f6): ``plane_lists`` puts every fitted track's registered mask on its registered
plane (``plane['fit']['reg_plane']``) and every other detection above the threshold on its own plane;
``plane_maps`` turns them into per-frame depth and surface-normal maps on the device (``engine.plane_maps``: the
nearest plane wins each pixel), and ``write_plane_maps`` writes them as 16-bit millimetre PNGs and a normal-map mp4
through the same chunked pipeline as ``write_video``.
"""
from __future__ import annotations

import os
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

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


def _stream_chunks(T: int, per: int, parts, produce, consume, device):
    """Bounded-chunk device -> host pipeline: ``produce(a, b)`` returns device tensors for frames [a, b) shaped
    like ``parts`` ((frame shape, dtype) each); they are copied into one of two sets of pinned host buffers, and
    ``consume(a, host tensors)`` runs on the host for a chunk while the device produces and copies the next."""
    with torch.cuda.device(device):
        pinned = [[torch.empty((per,) + tuple(shape), dtype=dt).pin_memory() for shape, dt in parts]
                  for _ in range(min(2, -(-T // per)))]
        pending = None
        for c, a in enumerate(range(0, T, per)):
            b = min(T, a + per)
            hosts = [buf[:b - a] for buf in pinned[c % 2]]
            for host, dev in zip(hosts, produce(a, b)):
                host.copy_(dev, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
            if pending is not None:
                pending[0].synchronize()
                consume(*pending[1:])              # the previous chunk, while this one is produced and copied
            pending = (done, a, hosts)
        if pending is not None:
            pending[0].synchronize()
            consume(*pending[1:])


def _video_writer(path: str, fps: float, W: int, H: int):
    import cv2
    writer = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (W, H))
    if not writer.isOpened():
        raise RuntimeError(f"cv2.VideoWriter cannot open {path}")
    return writer


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
    writer = _video_writer(path, fps, W, H)

    def encode(a, hosts):
        for frame in hosts[0].numpy():
            writer.write(cv2.cvtColor(frame, cv2.COLOR_RGB2BGR))

    try:
        _stream_chunks(T, per, [((H, W, 3), torch.uint8)],
                       lambda a, b: [_render_range(pool, lists, bg, a, b, device)], encode, device)
    finally:
        writer.release()
    return path


# ---------------------------------------------------------------------------
# depth and surface-normal maps of the fitted planes (row f6)
# ---------------------------------------------------------------------------
@dataclass
class PlaneLists:
    """Per-frame plane layers of a clip, indexing the same pool as ``DrawLists`` (``mask_pool`` builds it): the
    registered masks of every fitted track in track order, then every detection mask in (frame, box) order."""
    layers: np.ndarray           # _lib.PLANE_LAYER_DTYPE
    layer_begin: np.ndarray      # (T + 1,) int64
    fitted: list                 # plane dicts of the fitted tracks, in pool order
    n_reg: int                   # registered masks at the front of the pool


def normal_colours(normals) -> np.ndarray:
    """(n, 3) uint8 colours of fp32 unit normals: clamp(floor(127.5 (1 - n_i) + 0.5), 0, 255) in float64 (a NaN
    component gives 0).  A visible plane has n . ray > 0, so this colours the camera-facing normal -n."""
    n = np.asarray(normals, dtype=np.float32).astype(np.float64).reshape(-1, 3)
    c = np.floor(127.5 * (1.0 - n) + 0.5)
    return np.clip(np.nan_to_num(c, nan=0.0), 0, 255).astype(np.uint8)


def detection_planes(pred_planes) -> tuple[np.ndarray, np.ndarray]:
    """(normal (n, 3), offset (n,)) fp32 of detector plane rows, as ``geometry.source_geometry`` converts them:
    [a, b, c] -> [a, -c, b], normal = p / |p|, offset = |p|."""
    plane = torch.as_tensor(pred_planes).detach().cpu().to(torch.float32).clone().reshape(-1, 3)
    plane[:, [1, 2]] = plane[:, [2, 1]]
    plane[:, 1] = -plane[:, 1]
    return F.normalize(plane, p=2).numpy(), torch.norm(plane, p=2, dim=1).numpy()


def plane_lists(opt_preds, planes, cfg: OptConfig | None = None, score_thresh: float = 0.7) -> PlaneLists:
    """Plane layers of every frame of a clip (host only).  Per frame: every fitted track's registered mask on its
    ``fit['reg_plane']`` row, then every detection with score >= ``score_thresh`` whose box is not a fitted track's
    at that frame, on its own plane (``detection_planes``); each coloured by its normal (``normal_colours``)."""
    T = len(opt_preds)
    fitted = [pl for _, pl in _tracks(planes) if pl.get("has_rot", False)]
    rows = [[] for _ in range(T)]
    owned = set()
    base = 0
    for pl in fitted:
        reg = np.asarray(pl["fit"]["reg_plane"], dtype=np.float32).reshape(-1, 4)
        if len(reg) != len(pl["ids"]):
            raise ValueError(f"fit['reg_plane'] has {len(reg)} rows for {len(pl['ids'])} fitted frames")
        cols = normal_colours(reg[:, :3])
        for i, (f, b) in enumerate(pl["ids"].items()):
            rows[f].append((base + i, reg[i, :3], reg[i, 3], cols[i], 0))
            owned.add((int(f), int(b)))
        base += len(pl["ids"])
    n_reg = base
    for f, p in enumerate(opt_preds):
        scores = np.asarray(p.scores, dtype=np.float64).reshape(-1)
        keep = [int(b) for b in np.flatnonzero(scores >= score_thresh) if (f, int(b)) not in owned]
        if keep:
            normal, offset = detection_planes(torch.as_tensor(p.pred_planes)[keep])
            cols = normal_colours(normal)
            for i, b in enumerate(keep):
                rows[f].append((base + b, normal[i], offset[i], cols[i], 0))
        base += len(scores)
    layers, begin = _flatten(rows, _lib.PLANE_LAYER_DTYPE)
    return PlaneLists(layers, begin, fitted, n_reg)


def _plane_range(pool, lists: PlaneLists, cfg: OptConfig, a: int, b: int, device, bg_rgb=(0, 0, 0)):
    lb = lists.layer_begin
    return engine.plane_maps(pool, lists.layers[lb[a]:lb[b]], lb[a:b + 1] - lb[a], cfg, bg_rgb, device=device)


def plane_maps(opt_preds, planes, cfg: OptConfig | None = None, device=None, score_thresh: float = 0.7,
               bg_rgb=(0, 0, 0)):
    """(depth (T, H, W) fp32, rgb (T, H, W, 3) uint8) CUDA tensors of the clip's planes: every pixel's z of the
    nearest plane layer covering it (0 where none does) and that layer's normal colour (``bg_rgb`` where none)."""
    cfg = cfg or OptConfig()
    device = _device(device, planes)
    lists = plane_lists(opt_preds, planes, cfg, score_thresh)
    pool = mask_pool(opt_preds, lists, cfg, device)
    with torch.cuda.device(device):
        return _plane_range(pool, lists, cfg, 0, len(opt_preds), device)


def depth_millimetres(depth: torch.Tensor) -> torch.Tensor:
    """uint16 millimetres of fp32 metres as int16 bits (torch has no uint16 arithmetic):
    (z * 1000).round().clamp(0, 65535) in fp32 on the tensor's device; 0 = no plane."""
    mm = (depth * 1000.0).round_().clamp_(0, 65535).to(torch.int32)
    return mm.view(torch.int16).reshape(depth.shape + (2,))[..., 0].contiguous()     # low half, little endian


def write_plane_maps(out_dir: str, video_id: str, opt_preds, planes, fps: float = 30, cfg: OptConfig | None = None,
                     device=None, score_thresh: float = 0.7, chunk_bytes: int = 64 << 20) -> tuple[str, str]:
    """``plane_maps`` written as ``<out_dir>/<video_id>_depth/<k:05d>.png`` (uint16 millimetres, k = the frame's
    position in the clip) and ``<out_dir>/<video_id>_normals.mp4`` (cv2 ``mp4v``, black where no plane is).
    Chunks of at most ``chunk_bytes`` of depth + RGB go through pinned buffers as in ``write_video``.  Returns the
    directory and the video path."""
    import cv2
    cfg = cfg or OptConfig()
    H, W = cfg.height, cfg.width
    T = len(opt_preds)
    device = _device(device, planes)
    lists = plane_lists(opt_preds, planes, cfg, score_thresh)
    pool = mask_pool(opt_preds, lists, cfg, device)
    depth_dir = os.path.join(out_dir, f"{video_id}_depth")
    os.makedirs(depth_dir, exist_ok=True)
    path = os.path.join(out_dir, f"{video_id}_normals.mp4")
    per = max(1, min(T, chunk_bytes // (H * W * 5)))
    writer = _video_writer(path, fps, W, H)

    def produce(a, b):
        depth, rgb = _plane_range(pool, lists, cfg, a, b, device)
        return [depth_millimetres(depth), rgb]

    def encode(a, hosts):
        mm, rgb = hosts
        for i, (d, frame) in enumerate(zip(mm.numpy(), rgb.numpy())):
            if not cv2.imwrite(os.path.join(depth_dir, f"{a + i:05d}.png"), d.view(np.uint16)):
                raise RuntimeError(f"cv2.imwrite cannot write {depth_dir}/{a + i:05d}.png")
            writer.write(cv2.cvtColor(frame, cv2.COLOR_RGB2BGR))

    try:
        _stream_chunks(T, per, [((H, W), torch.int16), ((H, W, 3), torch.uint8)], produce, encode, device)
    finally:
        writer.release()
    return depth_dir, path
