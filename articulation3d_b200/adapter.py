"""Per-frame adapter either side of the hot path (SURVEY.md §8f rows f1, f2).

* ``create_instances`` — COCO-json detections -> ``Instances`` (reference
  utils/arti_vis.py:152-194).  ``masks='rle'`` keeps the run-length masks
  (``pred_rle``) so the optimizer decodes them on the device straight into packed
  bits; ``masks='dense'`` reproduces the reference's fp32 ``pred_masks``.
* ``override_depth`` — replaces every instance's plane offset by the mean over its
  mask of ``normal . XYZ`` (reference utils/arti_vis.py:125-149, with ``depth2XYZ``
  :90-99 and ``get_K_inv_dot_xy_1`` :101-122), as one device launch for all
  instances of all frames handed in; ``override_depth_records`` does the same for records carrying
  ``pred_depth``, streaming the depth through the device in bounded chunks.
* ``load_predictions`` / ``group_by_video`` — the ``instances_predictions.pth``
  record list of tools/opt_arti.py:56-76.
"""
from __future__ import annotations

import functools
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
    """All frames at once: one RLE decode launch + one masked-mean launch.  ``depths`` is (len(instances), H, W),
    ``xyzs`` one (3, H, W) map per frame and ``rays`` (3, H, W), with (H, W) the masks' size; other shapes are
    refused before any device use (the maps are indexed by frame position)."""
    if (depths is None) == (xyzs is None):
        raise ValueError("give exactly one of depths / xyzs")
    sizes = [det["segmentation"]["size"] for inst in instances for det in inst["instances"]]
    if sizes:
        H, W = (int(s) for s in sizes[0])
        maps = [("depths", depths, [len(instances), H, W]), ("rays", rays, [3, H, W])]
        if xyzs is not None:
            if len(xyzs) != len(instances):
                raise ValueError(f"{len(xyzs)} xyzs map(s) for {len(instances)} frame(s)")
            maps += [(f"xyzs[{f}]", x, [3, H, W]) for f, x in enumerate(xyzs)]
        for name, t, shape in maps:
            if t is not None and list(t.shape) != shape:
                raise ValueError(f"{name} has shape {list(t.shape)}, the masks need {shape}")
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
    pool = engine.rle_to_pool(rles, H, W, device)
    planes_t = torch.stack(planes).float()
    offset = torch.linalg.vector_norm(planes_t, dim=1)
    normal = planes_t / offset.clamp_min(1e-8)[:, None]
    idx = torch.arange(len(rles), dtype=torch.int32, device=device)
    if depths is not None:
        if rays is None:
            rays = torch.FloatTensor(get_K_inv_dot_xy_1(H, W)).to(device)
        off, cnt = engine.plane_offsets(pool, idx, normal.to(device), rays.to(device), depths.to(device),
                                        torch.tensor(frame_of, dtype=torch.int32, device=device))
    else:
        # one launch per distinct XYZ map (the reference signature hands in one frame at a time)
        off = torch.empty(len(rles), dtype=torch.float32, device=device)
        cnt = torch.empty(len(rles), dtype=torch.int32, device=device)
        fo = torch.tensor(frame_of, device=device)
        for f, xyz in enumerate(xyzs):
            sel = (fo == f).nonzero()[:, 0]
            if sel.numel():
                o, c = engine.plane_offsets(pool, idx[sel], normal[sel.cpu()].to(device), xyz.to(device))
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


@functools.lru_cache(maxsize=None)
def _depth_rays(H: int, W: int, device: torch.device) -> torch.Tensor:
    return torch.FloatTensor(get_K_inv_dot_xy_1(H, W)).to(device)


def check_depth_records(records):
    """Raise ``ValueError`` naming the record's ``file_name`` if a record carries no ``pred_depth``, if its
    ``pred_plane`` rows differ from its number of instances, or if its depth map is not the (H, W) of its masks'
    ``segmentation.size``.  Host-side only: no library load, no device use."""
    for r in records:
        name = r.get("file_name")
        if "pred_depth" not in r:
            raise ValueError(f"{name}: the record carries no pred_depth to override its planes from")
        n = len(r["instances"])
        if r["pred_plane"].dim() != 2 or r["pred_plane"].shape[0] != n:
            raise ValueError(f"{name}: pred_plane has shape {list(r['pred_plane'].shape)} for {n} instance(s)")
        sizes = {tuple(int(x) for x in d["segmentation"]["size"]) for d in r["instances"]}
        if len(sizes) > 1:
            raise ValueError(f"{name}: the masks mix frame sizes {sorted(sizes)}")
        if sizes and tuple(r["pred_depth"].shape) != next(iter(sizes)):
            raise ValueError(f"{name}: pred_depth has shape {list(r['pred_depth'].shape)}, "
                             f"the masks are {list(next(iter(sizes)))}")


def override_depth_records(records, device, chunk_bytes: int = 256 << 20):
    """``override_depth_batch`` of ``records`` (reference-format records carrying ``pred_depth``, possibly
    memory-mapped) with the depth streamed through the device in chunks, so device memory stays bounded by two
    chunks of depth plus one chunk's mask pool whatever the number of records.  Replaces every record's
    ``pred_plane`` in place, with the same quirks as ``override_depth_batch`` (the input plane tensor is swapped in
    place, an empty mask keeps its plane, records without instances pass through) and bit for bit the same values:
    ``k_plane_offsets`` reduces each instance in one CTA in a fixed order, so the chunking changes no value.

    Consecutive frames with instances form a chunk while their fp32 depth fits ``chunk_bytes`` (at least one
    frame) and their size does not change.  A chunk's depth maps are copied into one of two pinned staging
    blocks and sent on a side stream, so the copy of chunk k+1 runs while chunk k is decoded (one
    ``rle_to_pool``) and reduced (one ``plane_offsets``).  Offsets and counts stay on the device until one
    D2H copy at the end.  Every record is checked (``check_depth_records``) before any device work."""
    check_depth_records(records)
    device = torch.device(device)
    if device.type != "cuda":
        raise engine._lib.A3DError("override_depth needs a CUDA device (no CPU fallback)")
    planes = []
    for r in records:
        p = r["pred_plane"]
        p[:, [1, 2]] = p[:, [2, 1]]                     # in place, as the reference (:129-130)
        p[:, 1] = -p[:, 1]
        planes.append(p)
    frames = [r for r in records if r["instances"]]
    if not frames:
        return records
    planes_t = torch.cat(planes).float()
    offset = torch.linalg.vector_norm(planes_t, dim=1)
    normal = planes_t / offset.clamp_min(1e-8)[:, None]

    chunks, first = [], 0                               # (first frame, frames, first instance, instances, H, W)
    n_inst = 0
    for i, r in enumerate(frames):
        H, W = r["pred_depth"].shape
        if i > first and ((H, W) != tuple(chunks[-1][4:]) or (i - first + 1) * H * W * 4 > chunk_bytes):
            first = i
        if i == first:
            chunks.append([i, 0, n_inst, 0, H, W])
        chunks[-1][1] += 1
        chunks[-1][3] += len(r["instances"])
        n_inst += len(r["instances"])
    stage_elems = max(c[1] * c[4] * c[5] for c in chunks)

    with torch.cuda.device(device):
        main, side = torch.cuda.current_stream(), torch.cuda.Stream()
        normal_d = normal.to(device)
        pinned = [torch.empty(stage_elems, dtype=torch.float32, pin_memory=True) for _ in range(min(2, len(chunks)))]
        depth_d = [torch.empty(stage_elems, dtype=torch.float32, device=device) for _ in pinned]
        copied = [torch.cuda.Event() for _ in pinned]      # H2D of the slot's block done
        consumed = [None] * len(pinned)                     # launches reading the slot's device block enqueued

        def stage(k):
            s = k % len(pinned)
            f0, nf, _, _, H, W = chunks[k]
            copied[s].synchronize()                         # the block's previous H2D has read it
            host = pinned[s][:nf * H * W].view(nf, H, W)
            for j in range(nf):
                host[j].copy_(torch.as_tensor(frames[f0 + j]["pred_depth"]))
            with torch.cuda.stream(side):
                if consumed[s] is not None:
                    side.wait_event(consumed[s])
                depth_d[s][:nf * H * W].copy_(pinned[s][:nf * H * W], non_blocking=True)
                copied[s].record(side)

        parts_off, parts_cnt = [], []
        stage(0)
        for k, (f0, nf, i0, ni, H, W) in enumerate(chunks):
            if k + 1 < len(chunks):
                stage(k + 1)
            s = k % len(pinned)
            rles, frame_of = [], []
            for j in range(nf):
                for det in frames[f0 + j]["instances"]:
                    rles.append(det["segmentation"])
                    frame_of.append(j)
            pool = engine.rle_to_pool(rles, H, W, device)
            main.wait_event(copied[s])
            off, cnt = engine.plane_offsets(pool, torch.arange(ni, dtype=torch.int32, device=device),
                                            normal_d[i0:i0 + ni], _depth_rays(H, W, device),
                                            depth_d[s][:nf * H * W].view(nf, H, W),
                                            torch.tensor(frame_of, dtype=torch.int32, device=device))
            consumed[s] = torch.cuda.Event()
            consumed[s].record(main)
            parts_off.append(off)
            parts_cnt.append(cnt)
            del pool
        res = torch.cat([torch.cat(parts_off).view(torch.int32), torch.cat(parts_cnt)]).cpu()
    off, cnt = res[:n_inst].view(torch.float32), res[n_inst:]
    new = torch.where((cnt > 0)[:, None], normal * off[:, None], planes_t)       # empty mask keeps the plane
    new[:, [1, 2]] = new[:, [2, 1]]
    new[:, 2] = -new[:, 2]
    k = 0
    for r in frames:
        n = len(r["instances"])
        r["pred_plane"] = new[k:k + n].clone()
        k += n
    return records


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
