"""On-disk contracts of the temporal stage (SURVEY.md §8f rows f2, f3).

Input: the reference's ``instances_predictions.pth`` — a list of per-frame records
``{image_id, file_name, instances: [{image_id, category_id, bbox XYWH, score,
segmentation: COCO RLE}], pred_plane (n,3), pred_rot_axis (n,3), pred_tran_axis (n,2)
[, pred_depth (H,W)]}`` (writer: evaluation/arti_evaluation.py:153-180, reader:
tools/opt_arti.py:56-76).  Output: the optimised records tools/opt_arti.py:229-249
builds, plus the fitted per-track results (axis, angle-per-frame track) the reference
only holds implicitly, plus an optional Wavefront ``.obj`` of the articulated planes.
"""
from __future__ import annotations

import json
import os

import numpy as np
import torch

from . import adapter, geometry, rle
from .config import OptConfig


def preds_to_records(preds, video_id: str = "synthetic00_0_0", start_image_id: int = 0, device=None, depths=None):
    """list[Instances] (dense masks) -> list of reference-format records (RLE masks).  With a CUDA ``device`` the
    masks are thresholded (``> 0.5``), packed and encoded there, with the same records as a result.  ``depths``
    ((T,H,W), e.g. ``synth.render_depths``) is stored per frame as ``pred_depth`` (fp32, on the host)."""
    segs = None
    if device is not None:
        segs = iter(_encode_preds_on_device(preds, torch.device(device)))
    records = []
    for t, p in enumerate(preds):
        boxes = p.pred_boxes.tensor.numpy().astype(np.float64)
        inst = []
        for k in range(len(boxes)):
            x0, y0, x1, y1 = boxes[k].tolist()
            seg = next(segs) if segs is not None else rle.encode(p.pred_masks[k].numpy() > 0.5)
            inst.append({"image_id": start_image_id + t, "category_id": int(p.pred_classes[k]),
                         "bbox": [x0, y0, x1 - x0, y1 - y0], "score": float(p.scores[k]),
                         "segmentation": seg})
        records.append({"image_id": start_image_id + t, "file_name": f"{video_id}_{t}.png", "instances": inst,
                        "pred_plane": p.pred_planes.clone(), "pred_rot_axis": p.pred_rot_axis.clone(),
                        "pred_tran_axis": p.pred_tran_axis.clone()})
        if depths is not None:
            records[-1]["pred_depth"] = depths[t].to("cpu", torch.float32).clone()
    return records


def _encode_preds_on_device(preds, device) -> list:
    """RLE dicts of every instance mask of the clip (``pred_masks > 0.5``), frame by frame."""
    from . import engine
    n = sum(len(p.pred_masks) for p in preds)
    if n == 0:
        return []
    H, W = preds[0].pred_masks.shape[1:]
    pool = engine.PoolBuilder(n, H, W, device, thresh=0.5)
    with torch.cuda.device(device):
        for p in preds:
            if len(p.pred_masks):
                pool.append(p.pred_masks.to(device))
    return rle.bits_to_rles(pool.bits, H, W)


def records_to_preds(records, image_size=None, conf_threshold: float = 0.7, masks: str = "rle"):
    """Reference-format records of ONE video (in frame order) -> list[Instances]."""
    preds = []
    for r in records:
        size = image_size
        if size is None:
            size = tuple(r["instances"][0]["segmentation"]["size"]) if r["instances"] else (480, 640)
        preds.append(adapter.create_instances(r["instances"], size, pred_planes=r["pred_plane"].numpy(),
                                              pred_rot_axis=r["pred_rot_axis"], pred_tran_axis=r["pred_tran_axis"],
                                              conf_threshold=conf_threshold, masks=masks))
    return preds


def opt_preds_to_records(opt_preds, records):
    """Optimised Instances -> the records tools/opt_arti.py:229-249 appends to its output."""
    out = []
    for pred, r in zip(opt_preds, records):
        boxes = pred.pred_boxes.tensor.tolist()
        rec = {"image_id": r["image_id"], "file_name": r["file_name"], "instances": [],
               "pred_rot_axis": pred.pred_rot_axis, "pred_tran_axis": pred.pred_tran_axis,
               "pred_plane": pred.pred_planes}
        if "pred_depth" in r:
            rec["pred_depth"] = r["pred_depth"]
        for i, (x0, y0, x1, y1) in enumerate(boxes):
            rec["instances"].append({"image_id": r["image_id"], "category_id": pred.pred_classes[i],
                                     "bbox": [x0, y0, x1 - x0, y1 - y0], "score": pred.scores[i]})
        out.append(rec)
    return out


def tracks_summary(planes, masks: bool = False) -> list:
    """JSON-able fitted results per track: has_rot, std_axis, centre frame, R^2, and the
    angle-per-frame track (frame, angle index, angle value, inter, union, iou).  ``masks=True`` adds to every
    angle-track entry its registered mask (``plane['reg_masks']``) as COCO RLE, ``segmentation`` =
    ``{"size": [H, W], "counts": <ascii str>}``."""
    out = []
    for cat in ("trans", "rot"):
        for ti, plane in enumerate(planes[cat]):
            fit = plane.get("fit", {})
            rec = {"kind": cat, "track": ti, "frames": [int(f) for f in plane["ids"].keys()],
                   "boxes": [int(b) for b in plane["ids"].values()], "has_rot": bool(plane.get("has_rot", False)),
                   "rsq": [None if np.isnan(x) else float(x) for x in np.asarray(fit.get("rsq", []), dtype=np.float64)]}
            if rec["has_rot"]:
                rec["std_axis"] = torch.as_tensor(plane["std_axis"]).reshape(-1).tolist()
                rec["center_frame"] = int(fit["center_frame"])
                rec["angle_track"] = [
                    {"frame": int(f), "angle_id": int(a), "angle": float(v), "inter": int(i), "union": int(u),
                     "iou": None if np.isnan(o) else float(o)}
                    for f, a, v, i, u, o in zip(fit["frames"], fit["angle_id"], fit["angle"], fit["inter"],
                                                fit["union"], fit["iou"])]
                if masks:
                    segs = _reg_mask_rles(plane["reg_masks"])
                    for e in rec["angle_track"]:
                        seg = segs[e["frame"]]
                        e["segmentation"] = {"size": list(seg["size"]), "counts": seg["counts"].decode("ascii")}
            out.append(rec)
    return out


def _reg_mask_rles(reg_masks) -> dict:
    """frame -> RLE of the registered masks: on the device for the optimiser's packed ``RegMasks``, on the host
    for a plain mapping of dense masks."""
    if hasattr(reg_masks, "to_rle"):
        return reg_masks.to_rle()
    frames = list(reg_masks.keys())
    dense = np.stack([np.asarray(reg_masks[f]) for f in frames]) if frames else np.zeros((0, 1, 1), np.float32)
    return dict(zip(frames, rle.encode_many(dense)))


def save_results(out_dir: str, video_id: str, opt_records, planes, masks: bool = False):
    """``<video_id>_predictions_opt.pth`` (the records) and ``<video_id>_tracks.json`` (``tracks_summary``; with
    ``masks=True`` it carries the registered masks)."""
    os.makedirs(out_dir, exist_ok=True)
    torch.save(opt_records, os.path.join(out_dir, f"{video_id}_predictions_opt.pth"))
    with open(os.path.join(out_dir, f"{video_id}_tracks.json"), "w") as f:
        json.dump(tracks_summary(planes, masks=masks), f, indent=1)


def write_obj(path: str, preds, planes, frame: int, cfg: OptConfig | None = None):
    """Minimal Wavefront .obj of one frame's articulated planes: every tracked plane with a
    fitted axis becomes a quad (the mask's image-space bounding box unprojected onto its
    plane, utils/vis.py:86-102) and its 3-D articulation axis a line element.  Geometry only —
    the reference's textured, earcut-triangulated export (tools/inference.py:44-168) is
    visualisation and out of scope."""
    cfg = cfg or OptConfig()
    lines, nv = [f"# articulation3d_b200 frame {frame}"], 0
    for cat in ("trans", "rot"):
        for ti, plane in enumerate(planes[cat]):
            if not plane.get("has_rot") or frame not in plane["ids"]:
                continue
            b = plane["ids"][frame]
            p = preds[frame]
            geo = geometry.source_geometry(p, b, cfg, cat == "trans")
            x0, y0, x1, y1 = p.pred_boxes.tensor[b].tolist()
            quad = geometry.unproject_points([[x0, y0], [x1, y0], [x1, y1], [x0, y1]], geo.normal, geo.offset, cfg)
            lines.append(f"o {cat}{ti}")
            for v in quad:
                lines.append("v %.10f %.10f %.10f" % tuple(v))
            lines.append(f"f {nv + 1} {nv + 2} {nv + 3} {nv + 4}")
            nv += 4
            for v in geo.axis3d:
                lines.append("v %.10f %.10f %.10f" % tuple(v))
            lines.append(f"l {nv + 1} {nv + 2}")
            nv += 2
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    return nv
