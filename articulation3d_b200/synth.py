"""Synthetic detections for the temporal optimizer (SURVEY.md §8d scene generator).

There is no network, no dataset and no detector checkpoint, so benchmarks and
parity tests run on procedurally generated clips that satisfy the optimizer's
input contract (reference utils/arti_vis.py:152-194): per frame an ``Instances``
with ``scores, pred_boxes, pred_classes, pred_planes, pred_rot_axis,
pred_tran_axis, pred_masks``.

* rotation track ("door"): a planar quad hinged on a near-vertical 3-D line,
  opening angle linear in time; class 0; ``pred_rot_axis`` is the projected hinge
  expressed relative to the box centre.
* translation track ("drawer"): a quad sliding in its own plane; class 1;
  ``pred_tran_axis`` is the unit image direction of the slide.
* static track: a door that never moves (all fitted angles equal).
* jitter track: a door whose angle is uncorrelated with time (low R^2, expected
  ``has_rot == False``).

Masks are rendered by per-pixel ray/plane intersection plus an in-quad test,
written in torch so the same code runs on the CPU (tests, oracle) and on the GPU
(benchmarks at the 256-video scale).  Scene parameters always come from a CPU
generator, so a seed names the same scene on every device.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

from .axis import axis_to_angle_offset
from .config import OptConfig
from .structures import Boxes, Instances

KIND_ROT, KIND_TRANS, KIND_STATIC, KIND_JITTER = 0, 1, 2, 3


@dataclass
class VideoScene:
    """Per-track, per-frame geometry of one clip (CPU tensors, float64)."""
    kinds: torch.Tensor        # (N,) int
    hinge: torch.Tensor        # (N,T,3) a point of the quad's anchor edge
    d: torch.Tensor            # (N,3) unit direction of the anchor edge (hinge)
    w: torch.Tensor            # (N,T,3) unit in-plane direction across the quad
    width: torch.Tensor        # (N,)
    height: torch.Tensor       # (N,)
    slide: torch.Tensor        # (N,3) unit slide direction (translation tracks)
    morph: torch.Tensor        # (N,T) int in {-1,0,1}: erode / keep / dilate
    plane_jitter: torch.Tensor  # (N,T,3)
    box_jitter: torch.Tensor   # (N,T,4)
    n_frames: int


def _unit(v):
    return v / v.norm(dim=-1, keepdim=True)


def make_scene(seed: int, n_tracks: int, n_frames: int, cfg: OptConfig,
               kinds=None, static_frac: float = 0.2, trans_frac: float = 0.25) -> VideoScene:
    g = torch.Generator().manual_seed(int(seed))

    def U(lo, hi, *shape):
        return lo + (hi - lo) * torch.rand(*shape, generator=g, dtype=torch.float64)

    N, T = n_tracks, n_frames
    if kinds is None:
        r = torch.rand(N, generator=g)
        kinds = torch.where(r < static_frac, KIND_STATIC,
                            torch.where(r < static_frac + trans_frac, KIND_TRANS, KIND_ROT))
    kinds = torch.as_tensor(kinds, dtype=torch.int64)

    # image slots keep inter-track box IoU < 0.5
    cols = int(math.ceil(math.sqrt(N * cfg.width / cfg.height)))
    rows = int(math.ceil(N / cols))
    slot_w, slot_h = cfg.width / cols, cfg.height / rows
    f = cfg.focal_length

    depth = U(1.5, 3.0, N)
    slot = torch.arange(N)
    cxp = (slot % cols + 0.5) * slot_w + U(-0.05, 0.05, N) * slot_w
    cyp = (slot // cols + 0.5) * slot_h + U(-0.05, 0.05, N) * slot_h
    wpx = U(0.45, 0.8, N) * slot_w
    hpx = U(0.5, 0.85, N) * slot_h
    width = wpx * depth / f
    height = hpx * depth / f

    d = _unit(torch.stack([0.03 * torch.randn(N, generator=g, dtype=torch.float64),
                           torch.ones(N, dtype=torch.float64),
                           0.03 * torch.randn(N, generator=g, dtype=torch.float64)], 1))
    ex = torch.tensor([1.0, 0.0, 0.0], dtype=torch.float64).expand(N, 3)
    e1 = _unit(ex - (ex * d).sum(1, keepdim=True) * d)
    e2 = torch.cross(d, e1, dim=1)
    side = torch.where(torch.rand(N, generator=g) < 0.5, -1.0, 1.0).to(torch.float64)
    e1 = e1 * side[:, None]                  # hinge on the left or the right edge
    swing = torch.where(torch.rand(N, generator=g) < 0.5, -1.0, 1.0).to(torch.float64)

    # anchor edge: for side=+1 the quad spans [hinge, hinge + width*e1]
    xh = (cxp - cfg.cx) / f * depth - side * width / 2
    yh = (cyp - cfg.cy) / f * depth
    hinge0 = torch.stack([xh, yh, depth], 1)

    theta0 = U(-0.25, 0.25, N)
    theta_max = U(math.pi / 6, math.pi / 2, N)
    tt = torch.linspace(0, 1, T, dtype=torch.float64)
    theta = theta0[:, None] + theta_max[:, None] * tt[None, :]
    theta = torch.where((kinds == KIND_ROT)[:, None], theta, theta0[:, None].expand(N, T))
    noise = 0.6 * torch.rand(N, T, generator=g, dtype=torch.float64)
    theta = torch.where((kinds == KIND_JITTER)[:, None], theta0[:, None] + noise, theta)
    theta = theta * swing[:, None]
    w = torch.cos(theta)[..., None] * e1[:, None, :] + torch.sin(theta)[..., None] * e2[:, None, :]

    # translation tracks slide in their own plane along a mostly horizontal/vertical direction
    phi = U(-0.4, 0.4, N) + torch.where(torch.rand(N, generator=g) < 0.5, 0.0, math.pi / 2)
    w0 = w[:, 0, :]
    slide = _unit(torch.cos(phi)[:, None] * w0 + torch.sin(phi)[:, None] * d)
    speed = torch.where(kinds == KIND_TRANS, 0.012, 0.0).to(torch.float64)
    steps = (torch.arange(T, dtype=torch.float64) - (T - 1) / 2)
    hinge = hinge0[:, None, :] + (speed[:, None] * steps[None, :])[..., None] * slide[:, None, :]

    morph = torch.randint(-1, 2, (N, T), generator=g)
    plane_jitter = 0.02 * torch.randn(N, T, 3, generator=g, dtype=torch.float64)
    box_jitter = torch.randint(-2, 3, (N, T, 4), generator=g).to(torch.float64)
    return VideoScene(kinds, hinge, d, w, width, height, slide, morph, plane_jitter, box_jitter, T)


def render_track_masks(scene: VideoScene, track: int, cfg: OptConfig, device="cpu") -> torch.Tensor:
    """(T,H,W) bool masks of one track."""
    H, W, f = cfg.height, cfg.width, cfg.focal_length
    dt = torch.float32
    ys, xs = torch.meshgrid(torch.arange(H, device=device, dtype=dt),
                            torch.arange(W, device=device, dtype=dt), indexing="ij")
    rx = ((xs - cfg.cx) / f)[None]
    ry = ((ys - cfg.cy) / f)[None]
    h = scene.hinge[track].to(device=device, dtype=dt)          # (T,3)
    d = scene.d[track].to(device=device, dtype=dt)              # (3,)
    w = scene.w[track].to(device=device, dtype=dt)              # (T,3)
    n = torch.cross(d.expand_as(w), w, dim=1)                   # (T,3)
    off = (n * h).sum(1)                                        # (T,)
    denom = n[:, 0, None, None] * rx + n[:, 1, None, None] * ry + n[:, 2, None, None]
    t = off[:, None, None] / denom
    px, py, pz = t * rx - h[:, 0, None, None], t * ry - h[:, 1, None, None], t - h[:, 2, None, None]
    u = px * w[:, 0, None, None] + py * w[:, 1, None, None] + pz * w[:, 2, None, None]
    s = px * d[0] + py * d[1] + pz * d[2]
    wd, ht = float(scene.width[track]), float(scene.height[track])
    m = (t > 0) & (u >= 0) & (u <= wd) & (s >= -ht / 2) & (s <= ht / 2)
    # +-1 px morphology
    mf = m.to(dt)[:, None]
    dil = F.max_pool2d(mf, 3, 1, 1)[:, 0] > 0.5
    ero = F.max_pool2d(1 - mf, 3, 1, 1)[:, 0] < 0.5
    mo = scene.morph[track].to(device)[:, None, None]
    return torch.where(mo > 0, dil, torch.where(mo < 0, ero, m))


def _mask_boxes(masks: torch.Tensor) -> torch.Tensor:
    """(T,H,W) bool -> (T,4) float XYXY tight boxes (zeros for empty masks)."""
    T, H, W = masks.shape
    colany = masks.any(1)
    rowany = masks.any(2)
    xs = torch.arange(W, device=masks.device)
    ys = torch.arange(H, device=masks.device)
    big = 10 ** 6
    x0 = torch.where(colany, xs, big).min(1).values
    x1 = torch.where(colany, xs, -1).max(1).values + 1
    y0 = torch.where(rowany, ys, big).min(1).values
    y1 = torch.where(rowany, ys, -1).max(1).values + 1
    box = torch.stack([x0, y0, x1, y1], 1).to(torch.float64)
    box[x1 <= 0] = 0
    return box


def track_predictions(scene: VideoScene, track: int, cfg: OptConfig, masks: torch.Tensor,
                      frames=None):
    """Per-frame detector outputs of one track (CPU fp32 tensors):
    boxes (T,4), pred_planes (T,3), pred_rot_axis (T,3), pred_tran_axis (T,2).
    ``frames`` restricts the (python-loop) axis fields to those frames."""
    T = scene.n_frames
    f = cfg.focal_length
    boxes = _mask_boxes(masks).cpu() + scene.box_jitter[track]
    boxes[:, 0::2] = boxes[:, 0::2].clamp(0, cfg.width)
    boxes[:, 1::2] = boxes[:, 1::2].clamp(0, cfg.height)
    boxes = boxes.to(torch.float32)
    centers = (boxes[:, :2] + boxes[:, 2:]) / 2

    h, d, w = scene.hinge[track], scene.d[track], scene.w[track]
    n = torch.cross(d.expand_as(w), w, dim=1)
    n = _unit(n + scene.plane_jitter[track])
    off = (n * h).sum(1, keepdim=True)
    c = n * off                          # plane vector; invariant to the sign of n
    pred_planes = torch.stack([c[:, 0], c[:, 2], -c[:, 1]], 1).to(torch.float32)

    def proj(p):
        return torch.stack([f * p[:, 0] / p[:, 2] + cfg.cx, f * p[:, 1] / p[:, 2] + cfg.cy], 1)

    a, b = proj(h - 0.5 * d), proj(h + 0.5 * d)
    rot_axis = torch.zeros(T, 3)
    tran_axis = torch.zeros(T, 2)
    mid = h + 0.5 * scene.width[track] * w
    ta, tb = proj(mid), proj(mid + 0.1 * scene.slide[track])
    for t in (range(T) if frames is None else frames):
        line = [[float(a[t, 0]), float(a[t, 1]), float(b[t, 0]), float(b[t, 1])]]
        rot_axis[t] = axis_to_angle_offset(line, centers[t:t + 1])[0, :3]
        dxy = (tb[t] - ta[t])
        dxy = dxy / dxy.norm()
        tran_axis[t, 0] = float(dxy[0])      # direction of the line is (sin, -cos)
        tran_axis[t, 1] = float(-dxy[1])
    return boxes, pred_planes, rot_axis, tran_axis


def make_video(seed: int, n_tracks: int, n_frames: int, cfg: OptConfig | None = None,
               kinds=None, device="cpu", score: float = 0.95, drop_prob: float = 0.0,
               mask_dtype=torch.float32):
    """One synthetic clip -> (list[Instances] of length n_frames, VideoScene).

    ``drop_prob`` removes a detection from a frame with that probability (gaps in
    tracks, empty frames), exercising the tracker's gap logic."""
    cfg = cfg or OptConfig()
    scene = make_scene(seed, n_tracks, n_frames, cfg, kinds=kinds)
    g = torch.Generator().manual_seed(int(seed) + 7919)
    per_track = []
    for k in range(n_tracks):
        masks = render_track_masks(scene, k, cfg, device=device)
        boxes, planes, rot_axis, tran_axis = track_predictions(scene, k, cfg, masks)
        per_track.append((masks, boxes, planes, rot_axis, tran_axis))
    keep = torch.rand(n_tracks, n_frames, generator=g) >= drop_prob
    preds = []
    for t in range(n_frames):
        sel = [k for k in range(n_tracks) if bool(keep[k, t])]
        inst = Instances((cfg.height, cfg.width))
        inst.scores = np.full(len(sel), score, dtype=np.float64)
        inst.pred_boxes = Boxes(torch.stack([per_track[k][1][t] for k in sel])
                                if sel else torch.zeros(0, 4))
        inst.pred_classes = np.array([1 if int(scene.kinds[k]) == KIND_TRANS else 0 for k in sel],
                                     dtype=np.int64)
        inst.pred_planes = (torch.stack([per_track[k][2][t] for k in sel])
                            if sel else torch.zeros(0, 3))
        inst.pred_rot_axis = (torch.stack([per_track[k][3][t] for k in sel])
                              if sel else torch.zeros(0, 3))
        inst.pred_tran_axis = (torch.stack([per_track[k][4][t] for k in sel])
                               if sel else torch.zeros(0, 2))
        inst.pred_masks = (torch.stack([per_track[k][0][t] for k in sel]).to(mask_dtype)
                           if sel else torch.zeros(0, cfg.height, cfg.width, dtype=mask_dtype))
        preds.append(inst)
    return preds, scene


def scene_planes(scene: VideoScene) -> torch.Tensor:
    """(N,T,3) float64 true plane vectors ``n * offset`` of every track and frame, camera axes (x right, y down,
    z forward), without the detector's ``plane_jitter``."""
    n = torch.cross(scene.d[:, None, :].expand_as(scene.w), scene.w, dim=2)
    return n * (n * scene.hinge).sum(2, keepdim=True)


def scene_pred_planes(scene: VideoScene) -> torch.Tensor:
    """``scene_planes`` in the records' ``pred_plane`` axes (as ``track_predictions`` writes them), fp32."""
    c = scene_planes(scene)
    return torch.stack([c[..., 0], c[..., 2], -c[..., 1]], -1).to(torch.float32)


def render_depths(scene: VideoScene, cfg: OptConfig | None = None, device="cpu",
                  background: float = 10.0) -> torch.Tensor:
    """(T,H,W) fp32 depth maps of a clip, as the records' ``pred_depth``: every pixel's ray of the depth camera
    (``adapter.get_K_inv_dot_xy_1(H, W)``, z = 1) meets the true plane (``scene_planes``) of each track whose mask
    (``render_track_masks``) covers the pixel; the nearest intersection in front of the camera wins, and a pixel
    no track covers that way gets ``background``."""
    from .adapter import get_K_inv_dot_xy_1
    cfg = cfg or OptConfig()
    H, W = cfg.height, cfg.width
    rays = torch.from_numpy(get_K_inv_dot_xy_1(H, W)).to(device)                   # (3,H,W) float64
    planes = scene_planes(scene).to(device)                                         # (N,T,3)
    depth = torch.full((scene.n_frames, H, W), math.inf, dtype=torch.float64, device=device)
    for k in range(planes.shape[0]):
        masks = render_track_masks(scene, k, cfg, device=device)
        off = planes[k].norm(dim=1)                                                 # plane: normal . X = off
        normal = planes[k] / off[:, None]
        t = off[:, None, None] / torch.einsum("tc,chw->thw", normal, rays)
        hit = masks & (t > 0) & torch.isfinite(t)
        depth = torch.where(hit, torch.minimum(depth, t), depth)
    return torch.where(torch.isinf(depth), background, depth).to(torch.float32)


def clone_preds(preds, instances_cls=Instances, boxes_cls=Boxes):
    """Deep copy of a prediction list, optionally re-typed (e.g. into the shim
    classes the unmodified reference is run with)."""
    out = []
    for p in preds:
        q = instances_cls(p.image_size)
        q.scores = np.copy(p.scores)
        q.pred_boxes = boxes_cls(p.pred_boxes.tensor.clone())
        q.pred_classes = np.copy(p.pred_classes)
        q.pred_planes = p.pred_planes.clone()
        q.pred_rot_axis = p.pred_rot_axis.clone()
        q.pred_tran_axis = p.pred_tran_axis.clone()
        q.pred_masks = p.pred_masks.clone()
        out.append(q)
    return out
