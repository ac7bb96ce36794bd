"""Per-frame adapter either side of the hot path (SURVEY.md §8f rows f1, f2).

* ``create_instances`` — COCO-json detections -> ``Instances`` (reference
  utils/arti_vis.py:152-194).  ``masks='rle'`` keeps the run-length masks
  (``pred_rle``) so the optimizer decodes them on the device straight into packed
  bits; ``masks='dense'`` reproduces the reference's fp32 ``pred_masks``.
* ``override_depth`` — replaces every instance's plane offset by the mean over its
  mask of ``normal . XYZ`` (reference utils/arti_vis.py:125-149, with ``depth2XYZ``
  :90-99 and ``get_K_inv_dot_xy_1`` :101-122), as one device launch for all
  instances of all frames handed in.
* ``load_predictions`` / ``group_by_video`` — the ``instances_predictions.pth``
  record list of tools/opt_arti.py:56-76.
"""
from __future__ import annotations

import zipfile

import numpy as np
import torch

from . import engine, rle
from .structures import Boxes, Instances

DEPTH_FOCAL = 571.623718          # utils/arti_vis.py:101 (DeepV2D intrinsics), not get_pcd's 517.97
DEPTH_CX, DEPTH_CY = 319.5, 239.5


def get_K_inv_dot_xy_1(h: int = 480, w: int = 640, focal_length: float = DEPTH_FOCAL) -> np.ndarray:
    """(3, h, w) float64 table of K^-1 [xx, yy, 1] with xx = x/w*640, yy = y/h*480
    (reference utils/arti_vis.py:101-122, the double loop vectorised; every entry is the
    same 3-term dot product, evaluated left to right)."""
    K = np.array([[focal_length, 0, DEPTH_CX], [0, focal_length, DEPTH_CY], [0, 0, 1]])
    K_inv = np.linalg.inv(K)
    yy = (np.arange(h, dtype=np.float64) / h * 480)[:, None] * np.ones((1, w))
    xx = np.ones((h, 1)) * (np.arange(w, dtype=np.float64) / w * 640)[None, :]
    out = np.empty((3, h, w))
    for i in range(3):
        out[i] = (K_inv[i, 0] * xx + K_inv[i, 1] * yy) + K_inv[i, 2]
    return out


def _xywh_to_xyxy(b: np.ndarray) -> np.ndarray:
    b = b.astype(np.float64).copy()
    b[:, 2] += b[:, 0]
    b[:, 3] += b[:, 1]
    return b


def create_instances(predictions, image_size, pred_planes=None, pred_rot_axis=None, pred_tran_axis=None,
                     conf_threshold: float = 0.7, masks: str = "dense") -> Instances:
    """COCO-json detections of one frame -> Instances (boxes above ``conf_threshold``)."""
    ret = Instances(image_size)
    score = np.asarray([x["score"] for x in predictions])
    chosen = (score > conf_threshold).nonzero()[0]
    ret.scores = score[chosen]
    bbox = np.asarray([predictions[i]["bbox"] for i in chosen]).reshape(-1, 4)
    ret.pred_boxes = Boxes(torch.from_numpy(_xywh_to_xyxy(bbox)).float())
    ret.pred_classes = np.asarray([predictions[i]["category_id"] for i in chosen])
    if pred_planes is not None:
        ret.pred_planes = torch.FloatTensor(np.asarray([np.asarray(pred_planes[i]) for i in chosen]).reshape(-1, 3))
    if pred_rot_axis is not None:
        ret.pred_rot_axis = pred_rot_axis[chosen]
    if pred_tran_axis is not None:
        ret.pred_tran_axis = pred_tran_axis[chosen]
    rles = [predictions[i].get("segmentation") for i in chosen]
    if all(r is not None for r in rles):
        if masks == "rle":
            ret.pred_rle = list(rles)
        else:
            h, w = image_size
            dense = [rle.decode(r) for r in rles]
            ret.pred_masks = torch.FloatTensor(np.array(dense).reshape(-1, h, w))
    return ret


def override_depth(instance: dict, depth: torch.Tensor | None = None, xyz: torch.Tensor | None = None,
                   rays: torch.Tensor | None = None, device=None) -> dict:
    """Reference ``PlaneRCNN_Branch.override_depth(xyz, instance)`` for one frame record
    ``{'instances': [...COCO json with RLE...], 'pred_plane': (n,3) tensor}``; give either
    ``xyz`` (3,H,W) as the reference does, or ``depth`` (H,W) to fuse ``depth2XYZ``."""
    return override_depth_batch([instance], None if depth is None else depth[None],
                                None if xyz is None else [xyz], rays, device)[0]


def override_depth_batch(instances, depths: torch.Tensor | None = None, xyzs=None,
                         rays: torch.Tensor | None = None, device=None):
    """All frames at once: one RLE decode launch + one masked-mean launch."""
    if (depths is None) == (xyzs is None):
        raise ValueError("give exactly one of depths / xyzs")
    if device is None:
        device = (depths if depths is not None else xyzs[0]).device
    device = torch.device(device)
    if device.type != "cuda":
        raise engine._lib.A3DError("override_depth needs a CUDA device (no CPU fallback)")
    rles, frame_of, planes = [], [], []
    for f, inst in enumerate(instances):
        p = inst["pred_plane"]
        p[:, [1, 2]] = p[:, [2, 1]]                     # in place, as the reference (:129-130)
        p[:, 1] = -p[:, 1]
        for k, det in enumerate(inst["instances"]):
            rles.append(det["segmentation"])
            frame_of.append(f)
            planes.append(p[k])
    if not rles:
        return instances
    H, W = rles[0]["size"]
    pool = engine.rle_to_pool(rles, H, W, device)
    planes_t = torch.stack(planes).float()
    offset = torch.linalg.vector_norm(planes_t, dim=1)
    normal = planes_t / offset.clamp_min(1e-8)[:, None]
    idx = torch.arange(len(rles), dtype=torch.int32, device=device)
    if depths is not None:
        if rays is None:
            rays = torch.FloatTensor(get_K_inv_dot_xy_1(H, W)).to(device)
        off, cnt = engine.plane_offsets(pool, idx, normal.to(device), rays.to(device), depths.to(device).reshape(-1, H, W),
                                        torch.tensor(frame_of, dtype=torch.int32, device=device))
    else:
        # one launch per distinct XYZ map (the reference signature hands in one frame at a time)
        off = torch.empty(len(rles), dtype=torch.float32, device=device)
        cnt = torch.empty(len(rles), dtype=torch.int32, device=device)
        fo = torch.tensor(frame_of, device=device)
        for f, xyz in enumerate(xyzs):
            sel = (fo == f).nonzero()[:, 0]
            if sel.numel():
                o, c = engine.plane_offsets(pool, idx[sel], normal[sel.cpu()].to(device), xyz.to(device).reshape(3, H, W))
                off[sel], cnt[sel] = o, c
    off, cnt = off.cpu(), cnt.cpu()
    new = torch.where((cnt > 0)[:, None], normal * off[:, None], planes_t)       # empty mask keeps the plane
    new[:, [1, 2]] = new[:, [2, 1]]
    new[:, 2] = -new[:, 2]
    k = 0
    for inst in instances:
        n = len(inst["instances"])
        if n:
            inst["pred_plane"] = new[k:k + n].clone()
        k += n
    return instances


def load_predictions(path: str, mmap: bool = False):
    """``instances_predictions.pth``: list of per-keyframe dicts (tools/opt_arti.py:56-57).  ``mmap=True`` maps the
    tensors' storages from the file instead of reading them, so processes loading the same file share its pages;
    a file in torch's legacy (non-zip) format cannot be mapped and is read."""
    return torch.load(path, map_location="cpu", weights_only=False, mmap=mmap and zipfile.is_zipfile(path))


def video_key(file_name: str):
    """(video id, frame offset) of a record's file name ``<youtube id>_<shot>_<frame>_<offset>.png``:
    video id = ``{youtube_id}_{shot_id}_{frame_id}`` with the 11-character YouTube id, exactly as
    tools/opt_arti.py:60-76 builds it (two clips cut from the same YouTube video are two videos)."""
    stem = file_name.split('/')[-1].replace('.png', '')
    parts = stem.split('_')
    shot_id, frame_id, frame_offset = int(parts[-3]), int(parts[-2]), int(parts[-1])
    return '{}_{}_{}'.format(stem[:11], shot_id, frame_id), frame_offset


def group_by_video(predictions):
    """Records grouped per video id (``video_key``), each group ordered by frame offset; videos in
    order of first appearance (tools/opt_arti.py:60-76)."""
    out = {}
    for p in predictions:
        vid, off = video_key(p["file_name"])
        out.setdefault(vid, {})[off] = p            # a repeated offset replaces the record, as the reference's dict does
    return {vid: [frames[k] for k in sorted(frames)] for vid, frames in out.items()}
