"""Drop-in temporal articulation optimizer: ``track_planes`` / ``optimize_planes``.

Same names, argument meaning, return values, in-place side effects and global
``random`` consumption as the reference's utils/opt_utils.py (:962-974 dispatcher,
:382-682 ``optimize_planes_3dc``, :685-959 ``optimize_planes_3d_trans``,
:112-379 legacy ``'3d'``, :75-109 ``'average'``, :1156-1208 ``track_planes``),
with the pixel work moved to the device:

    reference (per source frame)                     here
    -------------------------------------------     ---------------------------------
    nonzero + get_pcd + Transform3d x A + project2D  a3d_project   (one launch per pass)
      + A python-loop scatters
    per target: >0.5, &, |, sum, sum, /, argmax      a3d_score     (one launch per pass)
    proj_masks[angle_id].cpu() per frame             lazy a3d_emit_masks

The control flow that depends on Python's global RNG and on list mutation
(SURVEY.md App. A #9, #11) is kept on the host, written once as a generator per
track list: it *yields* a job (source frame, candidate transforms, target frames)
and is *sent* the per-target arg-max back.  One video is driven job by job; many
videos are driven in lock-step so each device pass carries one job per video
(``optimize_videos``).

Additions over the reference (never removals): every optimised track gets
``plane['fit']`` — the per-frame angle index / inter / union / iou of the final
assignment, cluster R^2 values and the centre frame — i.e. the "angle-per-frame
track" the reference only holds implicitly; ``plane['reg_masks']`` is a lazy
mapping that materialises the fp32 masks on access instead of copying T x 1.2 MB
to the host eagerly.
"""
from __future__ import annotations

import os
import random as _global_random
import threading
from collections.abc import Mapping
from dataclasses import dataclass, field

import numpy as np
import torch
from scipy.stats import linregress as _scipy_linregress

# scipy wraps linregress in an axis/nan-policy decorator that costs more than the regression;
# for 1-D finite inputs it forwards unchanged to this inner function (tests/test_host_logic.py).
linregress = getattr(_scipy_linregress, "__wrapped__", _scipy_linregress)



_vecdot = getattr(np, "vecdot", None) or (lambda a, b: np.add.reduce(a * b))      # numpy < 2 has no vecdot
_installed_constant_r = None


def _constant_r_of_installed_scipy() -> float:
    """What ``scipy.stats.linregress`` of THIS environment returns as r for a constant series (NaN
    since scipy 1.9, 0.0 before): the default for ``OptConfig.constant_track_r``."""
    global _installed_constant_r
    if _installed_constant_r is None:
        import warnings
        with warnings.catch_warnings(), np.errstate(all="ignore"):
            warnings.simplefilter("ignore")
            _installed_constant_r = float(_scipy_linregress(range(5), np.full(5, 0.5)).rvalue)
    return _installed_constant_r


def _rvalue(y, constant_r: float | None = None) -> np.float64:
    """Pearson r of ``y`` against 0..n-1, exactly as ``scipy.stats.linregress(range(n), y).rvalue``
    computes it (float64; mean-removed dot products through ``np.vecdot``; clip to [-1, 1]) without the
    array-API plumbing around it, which costs several times the arithmetic.  The degenerate case
    (constant ``y``: zero variance and zero covariance) is ``constant_r`` — see
    ``OptConfig.constant_track_r``; None = the installed scipy's answer.  tests/test_host_logic.py checks
    bit equality with scipy."""
    y = np.asarray(y).astype(np.float64)
    n = y.shape[0]
    x = np.arange(n, dtype=np.float64)
    x_ = x - np.mean(x, keepdims=True)
    y_ = y - np.mean(y, keepdims=True)
    ssxm = _vecdot(x_, x_) / n
    ssym = _vecdot(y_, y_) / n
    ssxym = _vecdot(x_, y_) / n
    if ssxm == 0.0 or ssym == 0.0:
        if ssxym != 0:
            return np.float64(0.0)
        return np.float64(_constant_r_of_installed_scipy() if constant_r is None else constant_r)
    return np.clip(ssxym / np.sqrt(ssxm * ssym), -1.0, 1.0)


from . import _lib, engine, geometry
from .axis import angle_offset_to_axis, axis_to_angle_offset
from .config import OptConfig
from .structures import Instances as _OwnInstances
from .diagnostics import check_axis, check_monotonic, fit_plane_from_normals  # noqa: F401  (reference names, row a15)

__all__ = ["track_planes", "optimize_planes", "optimize_planes_3dc", "optimize_planes_3d_trans",
           "optimize_planes_3d", "optimize_planes_average", "optimize_videos", "RegMasks"]


# ---------------------------------------------------------------------------
# tracker (host only; reference utils/opt_utils.py:1156-1208)
# ---------------------------------------------------------------------------
def _box_iou_f32(a, b) -> float:
    """IoU of two XYXY boxes with every operation rounded to fp32, in the order
    detectron2's ``pairwise_iou`` evaluates it on 1x1 inputs (area1 + area2 - inter)."""
    f = np.float32
    iw = f(min(a[2], b[2]) - max(a[0], b[0]))
    ih = f(min(a[3], b[3]) - max(a[1], b[1]))
    if not (iw > 0 and ih > 0):
        return 0.0
    inter = f(iw * ih)
    area_a = f(f(a[2] - a[0]) * f(a[3] - a[1]))
    area_b = f(f(b[2] - b[0]) * f(b[3] - b[1]))
    return float(f(inter / f(f(area_a + area_b) - inter)))


def _box_iou_f32_arrays(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """``_box_iou_f32`` over broadcastable (..., 4) fp32 arrays: the same fp32 operations per pair."""
    with np.errstate(all="ignore"):
        iw = np.minimum(a[..., 2], b[..., 2]) - np.maximum(a[..., 0], b[..., 0])
        ih = np.minimum(a[..., 3], b[..., 3]) - np.maximum(a[..., 1], b[..., 1])
        inter = iw * ih
        area_a = (a[..., 2] - a[..., 0]) * (a[..., 3] - a[..., 1])
        area_b = (b[..., 2] - b[..., 0]) * (b[..., 3] - b[..., 1])
        iou = inter / ((area_a + area_b) - inter)
        return np.where((iw > 0) & (ih > 0), iou, np.float32(0.0)).astype(np.float32)


def track_planes(preds, cfg: OptConfig | None = None):
    """Greedy online box tracker -> {'rot': [...], 'trans': [...]}; each track is
    {'bbox', 'ids': {frame: box_id}, 'latest_frame'}.  A box joins the FIRST live
    track of its class (class 1 -> 'trans') whose latest box overlaps it with
    IoU > 0.5 and whose gap is <= 5 frames; tracks shorter than 10 frames are
    dropped (reference utils/opt_utils.py:1156-1208).

    A track's latest box is always a box of one of the last ``gap + 1`` frames (the current one
    included: a second box of a frame can match a track the first one just joined), so all box IoUs
    the greedy loop can ask for are evaluated up front in one fp32 array computation (the reference's
    operations per pair, same roundings) and the sequential part is list look-ups."""
    cfg = cfg or OptConfig()
    gap, thr = int(cfg.track_max_gap), cfg.track_iou
    T = len(preds)
    rows = [p.pred_boxes.tensor.detach().cpu().numpy().astype(np.float32, copy=False).reshape(-1, 4) for p in preds]
    counts = [len(r) for r in rows]
    nb = max(counts, default=0)
    planes = {'rot': [], 'trans': []}
    if nb:
        boxes = np.zeros((T, nb, 4), dtype=np.float32)
        for t, r in enumerate(rows):
            boxes[t, :len(r)] = r
        iou = []                                   # iou[d][t][i][j]: box i of frame t vs box j of frame t - d
        for d in range(min(gap, T - 1) + 1):
            m = np.zeros((T, nb, nb), dtype=np.float32)
            m[d:] = _box_iou_f32_arrays(boxes[d:, :, None, :], boxes[:T - d, None, :, :])
            iou.append(m.tolist())
        for idx in range(T):
            cls = np.asarray(preds[idx].pred_classes).reshape(-1).tolist()
            for box_id in range(counts[idx]):
                cat = 'trans' if cls[box_id] == 1 else 'rot'
                matched = False
                for plane in planes[cat]:
                    d = idx - plane['latest_frame']
                    if d > gap:
                        continue
                    if iou[d][idx][box_id][plane['_box']] > thr:
                        plane['ids'][idx] = box_id
                        plane['_box'] = box_id
                        plane['latest_frame'] = idx
                        matched = True
                        break
                if not matched:
                    planes[cat].append({'bbox': None, 'ids': {idx: box_id}, 'latest_frame': idx, '_box': box_id})
    for cat in planes:
        planes[cat] = [p for p in planes[cat] if len(p['ids']) >= cfg.track_min_len]
        for p in planes[cat]:
            p['bbox'] = preds[p['latest_frame']].pred_boxes[p.pop('_box')]
    return planes


# ---------------------------------------------------------------------------
# lazy reg_masks
# ---------------------------------------------------------------------------
class RegMasks(Mapping):
    """``plane['reg_masks']``: frame -> (H, W) fp32 CPU mask of the best candidate
    (reference utils/opt_utils.py:614, 906), unpacked from the device-resident
    bit-packed copy on first access."""

    def __init__(self, frames, packed: torch.Tensor, H: int, W: int):
        self._frames = list(frames)
        self._row = {f: i for i, f in enumerate(self._frames)}
        self.packed = packed            # (T, H, pitch) int32 on the device
        self._H, self._W = H, W
        self._cache = {}

    def __getitem__(self, frame):
        i = self._row[frame]
        if i not in self._cache:
            idx = torch.tensor([i], dtype=torch.int32, device=self.packed.device)
            self._cache[i] = engine.emit_masks(self.packed, idx, self._H, self._W)[0].cpu()
        return self._cache[i]

    def __iter__(self):
        return iter(self._frames)

    def __len__(self):
        return len(self._frames)

    def dense(self, dtype=torch.float32) -> torch.Tensor:
        """All masks as one (T, H, W) device tensor."""
        return engine.emit_masks(self.packed, None, self._H, self._W, dtype=dtype)

    def to_rle(self) -> dict:
        """frame -> COCO RLE dict of every mask, encoded on the device from the packed copy in one call (no dense
        image is made, nothing is cached)."""
        from . import rle
        return dict(zip(self._frames, rle.bits_to_rles(self.packed, self._H, self._W)))


# ---------------------------------------------------------------------------
# the host control flow, as a generator of device jobs
# ---------------------------------------------------------------------------
@dataclass
class SourceReq:
    """One cluster-round job whose source geometry is still to be computed (the driver batches the
    geometry of all pending requests into one set of array operations)."""
    frame: int                     # source frame
    box: int                       # its box
    translation: bool
    mode: int
    grid: object                   # candidate grid of the round (all requests of one kind share it)
    targets: list                  # pool indices, in id_list order


@dataclass
class JobSpec:
    source: int                    # pool index of the source mask
    mode: int
    normal: np.ndarray
    offset: float
    pivot: np.ndarray
    xform: np.ndarray              # (A, 12) fp32
    targets: list                  # pool indices, in id_list order
    keep_masks: bool = False       # final phase: return the winning packed masks


@dataclass
class JobResult:
    best_cand: np.ndarray          # (n_tgt,) int32
    best_iou: np.ndarray           # (n_tgt,) fp32
    best_inter: np.ndarray
    best_union: np.ndarray
    masks: torch.Tensor | None = None     # (n_tgt, H, pitch) int32 device, if keep_masks
    geo: "geometry.SourceGeometry | None" = None     # answer to a SourceReq: the source's geometry


@dataclass
class TrackTable:
    """Cluster-phase answers for EVERY frame of a track as source (all-sources schedule): row =
    source frame, column = target frame, both in ``frames`` order."""
    frames: list
    index: dict                    # frame -> row/column
    cand: np.ndarray               # (T, T) int32 first candidate of maximal IoU
    iou: np.ndarray                # (T, T) fp32 that IoU
    geo: "geometry.SourceGeometryRows"


@dataclass
class Stats:
    """What was evaluated, in the reference's accounting (BASELINE.md §3): one unit =
    one (visited frame, candidate) IoU."""
    units_visited: int = 0         # units the reference's loops evaluate
    units_computed: int = 0        # units the device evaluated
    passes: int = 0
    jobs: int = 0
    h2d_bytes: int = 0             # masks + job descriptors copied host -> device
    d2h_bytes: int = 0             # per-target results copied device -> host
    schedule: str = ""             # 'table' (all-sources pass + host replay) | 'chain' (a pass per round)
    detail: list = field(default_factory=list)


def _phase_setup(translation: bool, legacy: bool, cfg: OptConfig):
    if translation:
        return cfg.trans_grid, cfg.trans_grid, _lib.MODE_TRANSLATE, _lib.MODE_TRANSLATE
    if legacy:
        return cfg.legacy_grid, cfg.legacy_grid, _lib.MODE_SEQ, _lib.MODE_SEQ
    return cfg.rot_cluster_grid, cfg.rot_final_grid, _lib.MODE_SEQ, _lib.MODE_COMPOSED


def _angle_column(grid, mode: int) -> torch.Tensor:
    """The (A,1) fp32 tensor the reference indexes for a cluster's angle list."""
    if mode == _lib.MODE_TRANSLATE:
        return torch.as_tensor(grid, dtype=torch.float32).unsqueeze(1)
    return torch.FloatTensor(np.asarray(grid)[:, np.newaxis])


def _xforms_rows(dir_vec: np.ndarray, pivot: np.ndarray, grid, mode: int):
    """Candidate transforms of n sources at once: (n, A, 12) fp32 and R (n, A, 3, 3) or None."""
    if mode == _lib.MODE_TRANSLATE:
        return geometry.xforms_translate(grid, dir_vec), None
    if mode == _lib.MODE_SEQ:
        return geometry.xforms_seq_from_dirs(grid, dir_vec), None
    R = geometry.rotation_matrices(grid, dir_vec)
    return geometry.xforms_composed(R, pivot), R


class _VideoRows:
    """Per-box prediction rows of one video, flattened once so that the geometry of any set of
    (frame, box) sources is a gather plus one batched computation."""

    def __init__(self, preds):
        def flat(ts, width):
            ts = [t.detach().cpu().to(torch.float32).reshape(-1, width) for t in ts]
            return torch.cat(ts) if ts else torch.zeros(0, width)
        counts = [int(p.pred_boxes.tensor.shape[0]) for p in preds]
        self.base = np.zeros(len(preds) + 1, dtype=np.int64)
        np.cumsum(counts, out=self.base[1:])
        self.planes = flat([p.pred_planes for p in preds], 3)
        self.rot_axis = flat([p.pred_rot_axis for p in preds], 3)
        tran = flat([p.pred_tran_axis for p in preds], 2)
        self.tran_axis = torch.cat((tran, torch.zeros(len(tran), 1)), 1)      # offset column = 0
        boxes = flat([p.pred_boxes.tensor for p in preds], 4)
        self.centers = (boxes[:, :2] + boxes[:, 2:]) / 2

    def geometry(self, frames, boxes, translation: bool, cfg: OptConfig) -> geometry.SourceGeometryRows:
        idx = torch.from_numpy(self.base[np.asarray(frames, dtype=np.int64)] + np.asarray(boxes, dtype=np.int64))
        axis = self.tran_axis if translation else self.rot_axis
        return geometry.source_geometry_rows(self.planes[idx], axis[idx], self.centers[idx], cfg)


def _tracks_gen(preds, planes, cfg: OptConfig, translation: bool, rng, pool_of, stats: Stats,
                legacy: bool = False, tables=None):
    """Cluster rounds, model selection and final assignment for a list of tracks
    (reference :386-622 / :689-908 / legacy :113-340).  Mutates ``planes``.

    A cluster round needs, for its randomly chosen source frame, the arg-max candidate and IoU of
    every frame still in ``id_list``.  With ``tables`` (one ``TrackTable`` per track, computed for
    all sources in one device pass beforehand) the round is a table lookup and the generator only
    yields once, for the final-phase jobs; without, it yields a ``SourceReq`` per round and is sent
    a ``JobResult``."""
    cgrid, fgrid, cmode, fmode = _phase_setup(translation, legacy, cfg)
    remove_inliers = not legacy
    angles_c = _angle_column(cgrid, cmode)
    thr, n_cand = float(np.float32(cfg.inlier_iou)), len(cgrid)
    finals = []
    for ti, plane in enumerate(planes):
        ids = plane['ids']
        id_list = list(ids.keys())
        clusters = []
        geo_of = {}                       # source frame -> geometry (the final phase reuses its centre frame's)
        tab = tables[ti] if tables is not None else None
        for _ in range(cfg.rounds):
            if len(id_list) == 0 and remove_inliers:
                break
            select_idx = rng.choice(id_list)
            box_id = ids[select_idx]
            order = list(id_list)
            if tab is not None:
                r = tab.index[select_idx]
                cols = [tab.index[f] for f in order]
                ious, cands = tab.iou[r, cols].tolist(), tab.cand[r, cols].tolist()
            else:
                res = yield SourceReq(select_idx, box_id, translation, cmode, cgrid,
                                      [pool_of[(i, ids[i])] for i in order])
                geo_of[select_idx] = res.geo
                # plain python lists: fp32 IoUs are exact as doubles, so `> 0.5` decides as the fp32 compare does
                ious, cands = res.best_iou.tolist(), res.best_cand.tolist()
            row = {f: k for k, f in enumerate(order)}
            inliers, c_ids, c_ious = [], [], []
            it = 0
            while it < len(id_list):            # `for idx in id_list` with in-loop removal
                idx = id_list[it]
                it += 1
                k = row[idx]
                stats.units_visited += n_cand
                if ious[k] > thr:
                    inliers.append(idx)
                    if remove_inliers:
                        id_list.remove(idx)
                    c_ids.append(cands[k])
                    c_ious.append(ious[k])
            clusters.append({'center_id': select_idx, 'inliners': inliers,
                             'angles': angles_c[c_ids, 0].clone() if c_ids else torch.FloatTensor([]),
                             'ious': c_ious})

        rsqs = []
        for cluster in clusters:
            if len(cluster['inliners']) < cfg.min_inliers:
                rsqs.append(0.0)
                continue
            rsqs.append(_rvalue(cluster['angles'].numpy(), cfg.constant_track_r) ** 2)
        rsqs = np.array(rsqs)
        if rsqs.max() < cfg.rsq_thresh:
            plane['has_rot'] = False
            plane['fit'] = {'rsq': rsqs, 'clusters': clusters}
            continue
        plane['has_rot'] = True

        # final assignment: it draws no random numbers, so the final jobs of all tracks of this list
        # are deferred and scored together in ONE device pass after the last cluster round
        final_cluster = clusters[rsqs.argmax()]
        select_idx = final_cluster['center_id']
        box_id = ids[select_idx]
        p_instance = preds[select_idx]
        if legacy:
            geo = geometry.source_geometry(p_instance, box_id, cfg, translation, all_boxes=True)
        elif tab is not None:
            geo = tab.geo.row(tab.index[select_idx], box_id, int(p_instance.pred_boxes.tensor.shape[0]))
        else:
            geo = geo_of[select_idx]
        finals.append((plane, geo, select_idx, box_id, p_instance, rsqs, clusters))

    if not finals:
        return
    angles_f = _angle_column(fgrid, fmode)
    xf_all, R_all = _xforms_rows(np.stack([f[1].dir_vec for f in finals]), np.stack([f[1].pivot for f in finals]),
                                 fgrid, fmode)
    specs = []
    for k, (plane, geo, select_idx, box_id, p_instance, rsqs, clusters) in enumerate(finals):
        ids = plane['ids']
        specs.append(JobSpec(pool_of[(select_idx, box_id)], fmode, geo.normal.numpy(), float(geo.offset),
                             geo.pivot, xf_all[k], [pool_of[(i, b)] for i, b in ids.items()], keep_masks=True))
    results = yield specs
    H, W = cfg.height, cfg.width
    for k, ((plane, geo, select_idx, box_id, p_instance, rsqs, clusters), res) in enumerate(zip(finals, results)):
        frames = list(plane['ids'].keys())
        stats.units_visited += len(fgrid) * len(frames)
        plane['reg_masks'] = RegMasks(frames, res.masks, H, W)
        normal_trans = None
        if fmode == _lib.MODE_COMPOSED:
            normal_trans = geometry.transform_normals(geo.normal, R_all[k])
            sel = normal_trans[torch.from_numpy(res.best_cand.astype(np.int64))]
            sel = torch.stack((sel[:, 0], sel[:, 2], -sel[:, 1]), 1)          # [n0, n2, -n1]
            plane['reg_normals'] = dict(zip(frames, sel.unbind(0)))
        if translation:
            plane['std_axis'] = p_instance.pred_tran_axis[box_id]
        elif legacy:
            plane['std_axis'] = geo.pts.clone()
        else:
            plane['std_axis'] = geo.pts[box_id]
        plane['fit'] = {
            'frames': frames, 'center_frame': select_idx, 'rsq': rsqs, 'clusters': clusters,
            'angle_id': res.best_cand.copy(), 'angle': angles_f[:, 0].numpy()[res.best_cand],
            'inter': res.best_inter.copy(), 'union': res.best_union.copy(), 'iou': res.best_iou.copy(),
            # the plane of every fitted frame's registered mask, [n', d'] in get_pcd's camera frame
            'reg_plane': geometry.registered_planes(geo.normal, geo.offset, xf_all[k], fmode, geo.pivot,
                                                    res.best_cand, normals=normal_trans),
        }


# ---------------------------------------------------------------------------
# write-back (host; reference :624-682, :910-959, legacy :342-379)
# ---------------------------------------------------------------------------
def _rebuild(p_instance, scores):
    if type(p_instance) is _OwnInstances:          # same fields, same order, without eight length checks
        f = p_instance.get_fields()
        fields = {"scores": scores, "pred_boxes": f["pred_boxes"], "pred_planes": f["pred_planes"],
                  "pred_rot_axis": f["pred_rot_axis"], "pred_tran_axis": f["pred_tran_axis"]}
        for name in ("pred_masks", "pred_rle"):
            if name in f:
                fields[name] = f[name]
        fields["pred_classes"] = f["pred_classes"]
        out = _OwnInstances.__new__(_OwnInstances)
        object.__setattr__(out, "_image_size", p_instance.image_size)
        object.__setattr__(out, "_fields", fields)
        return out
    out = type(p_instance)(p_instance.image_size)
    out.scores = scores
    out.pred_boxes = p_instance.pred_boxes
    out.pred_planes = p_instance.pred_planes
    out.pred_rot_axis = p_instance.pred_rot_axis
    out.pred_tran_axis = p_instance.pred_tran_axis
    if _has(p_instance, 'pred_masks'):
        out.pred_masks = p_instance.pred_masks
    if _has(p_instance, 'pred_rle'):
        out.pred_rle = p_instance.pred_rle
    out.pred_classes = p_instance.pred_classes
    return out


def _has(p_instance, name: str) -> bool:
    return p_instance.has(name) if hasattr(p_instance, 'has') else hasattr(p_instance, name)


def _write_back(preds, planes, cfg: OptConfig, kind: str):
    """kind: 'rot' | 'trans' | 'legacy'.  The reference walks frames x tracks with one small tensor
    operation per (frame, track) (:624-682, :910-959); the arithmetic is elementwise fp32, so here all
    boxes of the video sit in flat arrays, every track is one gather / scatter, and the per-frame
    outputs are disjoint slices of those arrays (same values, same bits)."""
    n_frames = len(preds)
    counts = [int(p.pred_boxes.tensor.shape[0]) for p in preds]
    base = np.zeros(n_frames + 1, dtype=np.int64)
    np.cumsum(counts, out=base[1:])
    n = int(base[-1])
    classes = (np.concatenate([np.asarray(p.pred_classes).reshape(-1) for p in preds]) if n_frames
               else np.zeros(0, dtype=np.int64))
    if kind == 'legacy':
        chosen = np.zeros(n, dtype=bool)
    else:                                            # the other articulation type is never filtered
        chosen = classes == (1 if kind == 'rot' else 0)
    rot_axis = plane_rows = centers = None
    if kind == 'rot' and n_frames:
        rot_axis = torch.cat([p.pred_rot_axis for p in preds])          # new storage = the reference's clones
        plane_rows = torch.cat([p.pred_planes for p in preds])
        b = torch.cat([p.pred_boxes.tensor for p in preds])
        centers = (b[:, :2] + b[:, 2:]) / 2
    for plane in planes:
        ids = plane['ids']
        if not ids:
            continue
        rows = base[np.fromiter(ids.keys(), dtype=np.int64, count=len(ids))] + \
            np.fromiter(ids.values(), dtype=np.int64, count=len(ids))
        if not plane['has_rot']:
            chosen[rows] = False
            continue
        chosen[rows] = True
        if kind == 'rot':
            line = plane['std_axis'].unsqueeze(0).numpy().tolist()
            r = torch.from_numpy(rows)
            rot_axis[r] = axis_to_angle_offset(line * len(ids), centers[r])[:, :3]
        elif kind == 'trans':
            for f, bx in ids.items():
                preds[f].pred_tran_axis[bx] = plane['std_axis']     # in place, like the reference
    scores = (np.concatenate([np.asarray(p.scores).reshape(-1) for p in preds]) if n_frames
              else np.zeros(0))
    if scores.dtype.kind != 'f':
        scores = scores.astype(np.float64)
    decay = cfg.legacy_score_decay if kind == 'legacy' else cfg.score_decay
    scores[~chosen] = scores[~chosen] * decay
    opt_preds = []
    for idx, p_instance in enumerate(preds):
        lo, hi = int(base[idx]), int(base[idx + 1])
        if kind == 'rot':
            p_instance.pred_rot_axis = rot_axis[lo:hi]
            p_instance.pred_planes = plane_rows[lo:hi]
        opt_preds.append(_rebuild(p_instance, scores[lo:hi]))
    return opt_preds


# ---------------------------------------------------------------------------
# device session: mask pool + job driver
# ---------------------------------------------------------------------------
_UPLOAD_CHUNK_BYTES = 1 << 29      # dense masks staged on the device per pack call
_UPLOAD_DEPTH = 8                  # host -> device frame copies in flight (0 = no limit)
_PROJ_BUDGET_BYTES = 6 << 30       # projected-mask workspace of one device pass
_uploader = None                   # ONE helper thread: uploads of successive sessions queue up instead of sharing PCIe
_upload_streams: dict = {}         # device -> the stream all uploads of that device run on


def _upload_executor():
    global _uploader
    if _uploader is None:
        from concurrent.futures import ThreadPoolExecutor
        _uploader = ThreadPoolExecutor(max_workers=1, thread_name_prefix="a3d-upload")
    return _uploader


_preparer = None                   # ONE helper thread for the host-side preparation of the next video's table pass


def _prepare_executor():
    global _preparer
    if _preparer is None:
        from concurrent.futures import ThreadPoolExecutor
        _preparer = ThreadPoolExecutor(max_workers=1, thread_name_prefix="a3d-prepare")
    return _preparer


def _upload_stream(device) -> "torch.cuda.Stream":
    key = str(device)
    st = _upload_streams.get(key)
    if st is None:
        st = _upload_streams[key] = torch.cuda.Stream(device=device)
    return st


class _Session:
    """Packed masks of every tracked box of a set of videos, resident on one GPU."""

    def __init__(self, videos, cfg: OptConfig, device, ws=None, staging=None):
        self.cfg = cfg
        self.device = torch.device(device)
        self.ws = ws if ws is not None else engine.Workspace(self.device)        # shared by the sessions of a pipeline
        self.staging = staging if staging is not None else engine.Staging(self.device)
        self.videos = videos
        self.pool_of = []                   # per video: {(frame, box_id): pool index}
        self._rows = {}
        chunks, rles, n = [], [], 0
        for preds, plane_lists in videos:
            need = {}
            for planes in plane_lists:
                for plane in planes:
                    for f, b in plane['ids'].items():
                        need.setdefault(f, set()).add(b)
            index = {}
            for f in sorted(need):
                boxes = sorted(need[f])
                if _has(preds[f], 'pred_masks'):
                    m = preds[f].pred_masks
                    if tuple(m.shape[1:]) != (cfg.height, cfg.width):
                        raise ValueError(f"mask shape {tuple(m.shape[1:])} != camera {cfg.height}x{cfg.width}")
                    if len(boxes) == m.shape[0]:
                        chunks.append(m)
                    else:
                        # a frame with untracked boxes: runs of consecutive box ids as VIEWS of the frame's
                        # tensor.  (`m[boxes]` gathers into a fresh pageable tensor: a host copy per such frame
                        # plus a staged, synchronous transfer at a fifth of the pinned rate — 5-10 % of the
                        # frames of the synthetic clips, 10 of the 31 ms of a clip's upload.)
                        a = prev = boxes[0]
                        for b in boxes[1:]:
                            if b != prev + 1:
                                chunks.append(m[a:prev + 1])
                                a = b
                            prev = b
                        chunks.append(m[a:prev + 1])
                else:                        # run-length masks, decoded on the device
                    rles.extend(preds[f].pred_rle[b] for b in boxes)
                for b in boxes:
                    index[(f, b)] = n
                    n += 1
            self.pool_of.append(index)
        self.h2d_bytes = 0
        self.n_masks = n
        self._pool = None
        self._upload_future = self._upload_done = None
        if n == 0:
            return
        if rles:
            if chunks:
                raise ValueError("mixing dense pred_masks and pred_rle frames is not supported")
            self._pool = engine.rle_to_pool(rles, cfg.height, cfg.width, self.device)
            self.h2d_bytes += sum(len(r["counts"]) for r in rles)
            return
        self.h2d_bytes += sum(c.numel() * c.element_size() for c in chunks if not c.is_cuda)
        # The upload runs on its own stream from a helper thread, so the host-side preparation of the first
        # pass (source geometry, candidate transforms) and — with several videos — the device passes of the
        # previous video overlap the H2D copies, also when the driver makes the copy calls block.  One thread
        # and one stream for all sessions: the uploads of a pipeline of videos run one after the other at full
        # PCIe rate (two at once would both finish late).
        self._upload_stream = _upload_stream(self.device)
        self._upload_future = _upload_executor().submit(self._upload_worker, chunks, n)

    @property
    def pool(self):
        """The packed mask pool; the first access waits for the upload thread and orders the current
        stream after the upload stream."""
        if self._upload_future is not None:
            fut, self._upload_future = self._upload_future, None
            fut.result()                                   # re-raises what the upload thread raised
            torch.cuda.current_stream(self.device).wait_event(self._upload_done)
            for t in (self._pool.bits, self._pool.popc, self._pool.bbox) + tuple(self._pool._nz_pending or ()):
                t.record_stream(torch.cuda.current_stream(self.device))
        return self._pool

    def _upload_worker(self, chunks, n):
        torch.cuda.set_device(self.device)
        with torch.cuda.stream(self._upload_stream):
            self._pool = self._upload(chunks, n)
            self._upload_done = torch.cuda.Event()
            self._upload_done.record()
            # the next session's copies must not start before this one's are through (same stream: they do not),
            # and this thread returns only when they are, so that `pool` never waits on a half-filled stream
            self._upload_done.synchronize()
            self._upload_keep = None

    def _upload(self, chunks, n) -> engine.MaskPool:
        """Dense per-frame masks -> packed pool.  The frames are copied (asynchronously when the host
        tensors are pinned) into slices of ONE device staging block of at most _UPLOAD_CHUNK_BYTES and
        packed from there into the preallocated pool; no concatenated fp32 copy of all masks exists."""
        cfg = self.cfg
        H, W = cfg.height, cfg.width
        # mixed mask dtypes: everything is promoted to fp32 (never truncated to the first chunk's type)
        kinds = {c.dtype for c in chunks}
        if kinds <= {torch.uint8, torch.bool}:
            dt = torch.uint8
        else:
            dt = torch.float32
        per_mask = H * W * (4 if dt == torch.float32 else 1)
        cap = max(1, min(n, _UPLOAD_CHUNK_BYTES // per_mask))
        cap = max(cap, max(int(c.shape[0]) for c in chunks))
        builder = engine.PoolBuilder(n, H, W, self.device, with_nonzero=(dt == torch.float32),
                                     thresh=cfg.mask_thresh)
        stage = torch.empty(cap, H, W, dtype=dt, device=self.device)
        depth = int(os.environ.get("A3D_UPLOAD_DEPTH") or _UPLOAD_DEPTH)
        if all(not c.is_cuda for c in chunks) and os.environ.get("A3D_UPLOAD") != "python":
            # host masks: the whole loop below as ONE library call, outside the interpreter lock
            # (a3d_upload_masks, include/a3d.h)
            import ctypes as C
            cs = []
            for c in chunks:
                if c.dtype == torch.bool:
                    c = c.view(torch.uint8) if c.is_contiguous() else c.to(torch.uint8)
                if c.dtype != dt:
                    c = c.to(dt)
                cs.append(c.contiguous())
            self._upload_keep = cs                     # converted copies must outlive their transfers
            ptrs = (C.c_void_p * len(cs))(*[c.data_ptr() for c in cs])
            counts = (C.c_int64 * len(cs))(*[int(c.shape[0]) for c in cs])
            with torch.cuda.device(self.device):
                _lib.check(_lib.load().a3d_upload_masks(
                    ptrs, counts, len(cs), _lib.A3D_F32 if dt == torch.float32 else _lib.A3D_U8, H, W,
                    float(cfg.mask_thresh), stage.data_ptr(), cap, builder.bits.data_ptr(),
                    builder.nz.data_ptr() if builder.nz is not None else None, depth,
                    torch.cuda.current_stream().cuda_stream), "a3d_upload_masks")
            builder.fill = n
            return builder.finish()
        fill = 0
        # At most `depth` frame copies are in flight.  Submitted all at once (120 copies, 1.2 GB per clip) they
        # fill the copy engine's queue, the submitting call then blocks INSIDE the driver, and every other
        # thread's next CUDA call — the launch of the previous video's table pass — waits for it: 14 ms per
        # video (tools/e2e_timeline.py).
        inflight = []
        for c in chunks:
            if c.dtype == torch.bool:
                c = c.view(torch.uint8) if c.is_contiguous() else c.to(torch.uint8)
            if c.dtype != dt:
                c = c.to(dt)
            k = int(c.shape[0])
            if fill + k > cap:
                builder.append(stage[:fill])
                fill = 0
            stage[fill:fill + k].copy_(c, non_blocking=True)
            fill += k
            if depth > 0 and not c.is_cuda:
                ev = torch.cuda.Event()
                ev.record()
                inflight.append(ev)
                if len(inflight) > depth:
                    inflight.pop(0).synchronize()
        if fill:
            builder.append(stage[:fill])
        return builder.finish()

    def rows(self, v: int) -> _VideoRows:
        r = self._rows.get(v)
        if r is None:
            r = self._rows[v] = _VideoRows(self.videos[v][0])
        return r

    # -- device passes ------------------------------------------------------------------
    def _pass(self, batch: engine.JobBatch, host_out: np.ndarray | None, stats: Stats | None):
        """One device pass; the (4, n_tgt) result block is copied into pinned memory (D2H enqueued,
        not waited for).  Returns (PassResult, pinned int32 tensor view)."""
        dbatch = engine.DeviceBatch(batch, self.device, self.staging, self.cfg)
        res = engine.run_pass(self.cfg, self.pool, dbatch, self.ws)
        if stats is not None:
            stats.passes += 1
            stats.jobs += batch.n_jobs
            stats.units_computed += batch.units
            stats.h2d_bytes += batch.jobs.nbytes + batch.xform.nbytes + batch.tgt_index.nbytes
            stats.d2h_bytes += 16 * len(batch.tgt_index)
        return res

    def run(self, specs, stats: Stats | None = None):
        """One device pass over a list of JobSpec -> list of JobResult."""
        batch = engine.build_batch([s.source for s in specs], [s.mode for s in specs],
                                   [s.normal for s in specs], [s.offset for s in specs],
                                   [s.pivot for s in specs], [s.xform for s in specs],
                                   [s.targets for s in specs], self.pool.source_points)
        res = self._pass(batch, None, stats)
        host = self.staging.results_host(res.block.numel())
        host.view(4, -1).copy_(res.block, non_blocking=True)                 # one D2H into pinned memory
        # the winning masks of all jobs that keep theirs: ONE gather into ONE block (enqueued before the sync, so
        # it overlaps the D2H); the jobs' RegMasks hold views of it.  (A block per job was a fresh cudaMalloc per
        # track — the blocks stay alive with the results — and cost more than the final pass itself.)
        masks, keep = {}, [j for j, s in enumerate(specs) if s.keep_masks]
        if keep:
            spans, parts, o = {}, [], 0
            for j in keep:
                a, n = int(batch.jobs[j]["tgt_begin"]), int(batch.jobs[j]["n_tgt"])
                parts.append(res.best_cand[a:a + n] + int(batch.jobs[j]["cand_begin"]))
                spans[j] = (o, o + n)
                o += n
            block = res.masks(torch.cat(parts) if len(parts) > 1 else parts[0])      # copy out of the workspace
            masks = {j: block[lo:hi] for j, (lo, hi) in spans.items()}
        torch.cuda.current_stream().synchronize()
        packed = host.numpy().reshape(4, -1)
        out = []
        for j, s in enumerate(specs):
            a, n = int(batch.jobs[j]["tgt_begin"]), int(batch.jobs[j]["n_tgt"])
            out.append(JobResult(packed[0, a:a + n].copy(), packed[3, a:a + n].copy().view(np.float32),
                                 packed[1, a:a + n].copy(), packed[2, a:a + n].copy(), masks.get(j)))
        return out

    def run_rows(self, sources, modes, geo: geometry.SourceGeometryRows, xform, n_tgt, tgt_index,
                 stats: Stats | None = None, wait: bool = True):
        """Jobs given as arrays (one row of ``geo`` / ``xform[i]`` per job) -> (4, sum n_tgt) int32
        results {cand, inter, union, iou bits}.  Split into as many device passes as the
        projected-mask workspace budget asks for; all passes are enqueued before the one sync.
        ``wait=False``: nothing is waited for — returns (pinned int32 tensor of its own, event)."""
        S = len(sources)
        n_tgt = np.asarray(n_tgt, dtype=np.int64)
        A = xform.shape[1]
        per_cand = self.cfg.height * _lib.pitch_words(self.cfg.width) * 4
        per_pass = max(1, int(_PROJ_BUDGET_BYTES // (per_cand * max(A, 1))))
        t_begin = np.zeros(S + 1, dtype=np.int64)
        np.cumsum(n_tgt, out=t_begin[1:])
        total = 4 * int(t_begin[-1])
        host = (self.staging.results_host(total) if wait else torch.empty(max(total, 1), dtype=torch.int32).pin_memory()[:total])
        host = host.view(4, -1)
        src_points = self.pool.source_points
        for lo in range(0, S, per_pass):
            hi = min(S, lo + per_pass)
            batch = engine.build_batch_rows(sources[lo:hi], modes[lo:hi], geo.normal[lo:hi], geo.offset[lo:hi],
                                            geo.pivot[lo:hi], xform[lo:hi].reshape(-1, 12),
                                            np.full(hi - lo, A), tgt_index[t_begin[lo]:t_begin[hi]],
                                            n_tgt[lo:hi], src_points)
            res = self._pass(batch, None, stats)
            # row by row: a column slice of the (4, n) block is strided, and a strided device -> host copy is
            # staged through a temporary and WAITED for (the host then sat out the whole table pass here)
            for r in range(4):
                host[r, t_begin[lo]:t_begin[hi]].copy_(res.block[r], non_blocking=True)
        if not wait:
            done = torch.cuda.Event()
            done.record()
            return host, done
        torch.cuda.current_stream().synchronize()
        return host.numpy()

    # -- all-sources schedule -----------------------------------------------------------
    def _prepare_groups(self, lists, legacy: bool = False):
        """Host half of ``cluster_tables``: for all tracks of ``lists`` the geometry of every frame as a source,
        its candidate transforms and the job arrays — CPU work only (no access to the mask pool), so a helper
        thread can run it while the video's masks are still being uploaded and the previous video is optimised."""
        cfg = self.cfg
        groups = {}                                   # translation flag -> per-track bookkeeping
        for li, (v, planes, translation) in enumerate(lists):
            for ti, plane in enumerate(planes):
                frames = list(plane['ids'].keys())
                boxes = [plane['ids'][f] for f in frames]
                groups.setdefault(bool(translation), []).append((li, ti, v, frames, boxes))
        prepared = []
        for translation, tracks in groups.items():
            cgrid, _, cmode, _ = _phase_setup(translation, legacy, cfg)
            by_video = {}
            for k, (li, ti, v, frames, boxes) in enumerate(tracks):
                by_video.setdefault(v, []).append(k)
            # geometry of all sources: one batched computation per video's rows
            geo_of_track = [None] * len(tracks)
            for v, ks in by_video.items():
                fr = np.concatenate([np.asarray(tracks[k][3], dtype=np.int64) for k in ks])
                bx = np.concatenate([np.asarray(tracks[k][4], dtype=np.int64) for k in ks])
                g = self.rows(v).geometry(fr, bx, translation, cfg)
                o = 0
                for k in ks:
                    T = len(tracks[k][3])
                    geo_of_track[k] = (g, o, o + T)
                    o += T
            # one job list over all tracks, in track order
            src, ntg, tgt, parts = [], [], [], []
            for k, (li, ti, v, frames, boxes) in enumerate(tracks):
                pool_of = self.pool_of[v]
                tpool = np.fromiter((pool_of[(f, b)] for f, b in zip(frames, boxes)), dtype=np.int32,
                                    count=len(frames))
                T = len(frames)
                src.append(tpool.astype(np.int64))
                ntg.append(np.full(T, T, dtype=np.int64))
                tgt.append(np.tile(tpool, T))
                g, a, b = geo_of_track[k]
                parts.append(geometry.SourceGeometryRows(g.normal[a:b], g.offset[a:b], g.pts[a:b], g.axis3d[a:b],
                                                         g.dir_vec[a:b], g.pivot[a:b]))
            geo = geometry.concat_rows(parts)
            xform, _ = _xforms_rows(geo.dir_vec, geo.pivot, cgrid, cmode)
            prepared.append((tracks, parts, geo, xform, np.concatenate(src), np.concatenate(ntg), np.concatenate(tgt), cmode))
        return prepared

    def prefetch_tables(self, lists, legacy: bool = False):
        """Start ``_prepare_groups(lists)`` on the preparation thread; ``cluster_tables`` of the same lists
        picks the result up."""
        self._prep_key = (tuple((v, id(planes), bool(t)) for v, planes, t in lists), legacy)
        self._prep_future = _prepare_executor().submit(self._prepare_groups, lists, legacy)

    def launch_tables(self, lists, stats: Stats | None = None, legacy: bool = False):
        """First half of ``cluster_tables``: enqueues the all-sources pass(es) of ``lists`` and the D2H of
        their result blocks, waits for nothing on the device.  ``finish_tables`` turns the handle into tables."""
        key = (tuple((v, id(planes), bool(t)) for v, planes, t in lists), legacy)
        fut, self._prep_future = getattr(self, "_prep_future", None), None
        if fut is not None and getattr(self, "_prep_key", None) == key:
            prepared = fut.result()
        else:
            prepared = self._prepare_groups(lists, legacy)
        pending = []
        for tracks, parts, geo, xform, src, ntg, tgt, cmode in prepared:
            host, done = self.run_rows(src, np.full(len(src), cmode, dtype=np.int32), geo, xform, ntg, tgt, stats,
                                       wait=False)
            pending.append((tracks, parts, host, done))
        return key, [len(planes) for _, planes, _ in lists], pending

    @staticmethod
    def finish_tables(handle):
        _, sizes, pending = handle
        out = [[None] * n for n in sizes]
        for tracks, parts, host, done in pending:
            done.synchronize()
            res = host.numpy()
            o = 0
            for k, (li, ti, v, frames, boxes) in enumerate(tracks):
                T = len(frames)
                blk = res[:, o:o + T * T]
                out[li][ti] = TrackTable(frames, {f: i for i, f in enumerate(frames)},
                                         blk[0].reshape(T, T).copy(), blk[3].view(np.float32).reshape(T, T).copy(),
                                         parts[k])
                o += T * T
        return out

    def cluster_tables(self, lists, stats: Stats | None = None, legacy: bool = False):
        """``lists``: [(video index, planes, translation)].  ONE scheduling step for the cluster phase of
        all those track lists: every frame of every track is a source (job), its targets are all
        frames of its track.  Returns one list of ``TrackTable`` per entry of ``lists``."""
        return self.finish_tables(self.launch_tables(lists, stats, legacy))


def _table_units(lists, cfg: OptConfig) -> int:
    """Device work of the all-sources schedule for these track lists, in units."""
    u = 0
    for _, planes, translation in lists:
        a = len(cfg.trans_grid) if translation else len(cfg.rot_cluster_grid)
        u += sum(len(p['ids']) ** 2 for p in planes) * a
    return u


def _answer_chain(session: _Session, reqs, stats: Stats):
    """Chained schedule: one device pass for the pending requests of all generators.  ``reqs`` is a
    list of (video index, SourceReq | [JobSpec]); returns the answers in order."""
    cfg = session.cfg
    answers = [None] * len(reqs)
    # final-phase job lists go through the per-spec path (few jobs, winning masks kept)
    spec_jobs = [(i, r) for i, (_, r) in enumerate(reqs) if isinstance(r, list)]
    src_jobs = [(i, v, r) for i, (v, r) in enumerate(reqs) if not isinstance(r, list)]
    if src_jobs:
        # geometry of all pending sources, batched per (video, kind); jobs keep request order
        geo_rows = [None] * len(src_jobs)
        by = {}
        for k, (i, v, r) in enumerate(src_jobs):
            by.setdefault((v, r.translation), []).append(k)
        for (v, translation), ks in by.items():
            g = session.rows(v).geometry([src_jobs[k][2].frame for k in ks], [src_jobs[k][2].box for k in ks],
                                         translation, cfg)
            for j, k in enumerate(ks):
                geo_rows[k] = (g, j)
        for translation in (True, False):
            ks = [k for k, (i, v, r) in enumerate(src_jobs) if r.translation == translation]
            if not ks:
                continue
            mode, grid = src_jobs[ks[0]][2].mode, src_jobs[ks[0]][2].grid
            parts = []
            for k in ks:
                g, j = geo_rows[k]
                parts.append(geometry.SourceGeometryRows(g.normal[j:j + 1], g.offset[j:j + 1], g.pts[j:j + 1],
                                                         g.axis3d[j:j + 1], g.dir_vec[j:j + 1], g.pivot[j:j + 1]))
            geo = geometry.concat_rows(parts)
            xform, _ = _xforms_rows(geo.dir_vec, geo.pivot, grid, mode)
            src = np.array([session.pool_of[src_jobs[k][1]][(src_jobs[k][2].frame, src_jobs[k][2].box)] for k in ks],
                           dtype=np.int64)
            ntg = np.array([len(src_jobs[k][2].targets) for k in ks], dtype=np.int64)
            tgt = np.concatenate([np.asarray(src_jobs[k][2].targets, dtype=np.int32) for k in ks])
            res = session.run_rows(src, np.full(len(ks), mode, dtype=np.int32), geo, xform, ntg, tgt, stats)
            o = 0
            for j, k in enumerate(ks):
                i, v, r = src_jobs[k]
                n = int(ntg[j])
                n_boxes = int(session.videos[v][0][r.frame].pred_boxes.tensor.shape[0])
                answers[i] = JobResult(res[0, o:o + n].copy(), res[3, o:o + n].copy().view(np.float32),
                                       res[1, o:o + n].copy(), res[2, o:o + n].copy(),
                                       geo=geo.row(j, r.box, n_boxes))
                o += n
    if spec_jobs:
        flat, spans = [], []
        for i, specs in spec_jobs:
            spans.append((i, len(flat), len(specs)))
            flat.extend(specs)
        results = session.run(flat, stats)
        for i, lo, n in spans:
            answers[i] = results[lo:lo + n]
    return answers


def _drive(gens, session: _Session, stats: Stats, video_of=None):
    """Run generators in lock-step: every scheduling step carries the pending request of each
    still-active generator (``video_of[i]`` = video index of generator i)."""
    video_of = video_of or [0] * len(gens)
    pending = {}
    for i, g in enumerate(gens):
        try:
            pending[i] = next(g)
        except StopIteration:
            pass
    while pending:
        keys = list(pending.keys())
        answers = _answer_chain(session, [(video_of[k], pending[k]) for k in keys], stats)
        for k, ans in zip(keys, answers):
            try:
                pending[k] = gens[k].send(ans)
            except StopIteration:
                del pending[k]


def _use_tables(lists, cfg: OptConfig) -> bool:
    """Schedule choice.  'table': the cluster phase of every track is answered from one all-sources
    device pass (T x more device work, no host<->device round trip per round) — right when the rounds'
    latency dominates, and whenever the masks arrive as dense host arrays (their H2D copy then costs more
    than the table pass, which hides behind it).  'chain': one pass per round carrying one job per
    video — right for big batches of cheap inputs, where the device work dominates."""
    mode = os.environ.get("A3D_SCHEDULE") or cfg.schedule
    if mode == "table":
        return True
    if mode == "chain":
        return False
    return _table_units(lists, cfg) <= cfg.table_max_units


def _default_device(device):
    if device is not None:
        return torch.device(device)
    if not torch.cuda.is_available():
        raise _lib.A3DError("articulation3d_b200 needs a CUDA device; there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


# ---------------------------------------------------------------------------
# public API (reference signatures)
# ---------------------------------------------------------------------------
def _table_lists(video_lists):
    return [(v, planes, translation) for v, stages in enumerate(video_lists)
            for (_, planes, translation, _, _) in stages if planes]


def _run_lists(session: _Session, video_lists, cfg: OptConfig, stats: Stats, legacy: bool = False,
               use_tables: bool | None = None, launched=None):
    """Drive track lists to completion.  ``video_lists``: per video a list of stages
    ``(preds_fn, planes, translation, rng, after)``; the stages of a video run in order (their RNG
    consumption is sequential), videos advance in lock-step.  ``preds_fn()`` gives the stage's input
    predictions, ``after()`` is called when the stage is done (write-back)."""
    lists = _table_lists(video_lists)
    tables = {}
    if lists and session.n_masks and (use_tables if use_tables is not None else _use_tables(lists, cfg)):
        stats.schedule = "table"
        # ``launched``: the all-sources passes of these lists were already enqueued (optimize_videos does that
        # one video ahead, so the device works on them while the host replays the previous video)
        got = session.finish_tables(launched) if launched is not None else session.cluster_tables(lists, stats, legacy=legacy)
        for (v, planes, translation), tabs in zip(lists, got):
            tables[(v, translation)] = tabs
    elif lists:
        stats.schedule = "chain"

    def video_gen(v, stages):
        for preds_fn, planes, translation, rng, after in stages:
            yield from _tracks_gen(preds_fn(), planes, cfg, translation, rng, session.pool_of[v], stats,
                                   legacy=legacy, tables=tables.get((v, translation)))
            after()

    _drive([video_gen(v, stages) for v, stages in enumerate(video_lists)], session, stats,
           video_of=list(range(len(video_lists))))


def optimize_planes_3d_trans(preds, planes, frames=None, cfg=None, device=None, rng=None,
                             _session=None, stats=None):
    """Translation tracks (reference utils/opt_utils.py:685-959)."""
    cfg, stats = cfg or OptConfig(), stats if stats is not None else Stats()
    session = _session or _Session([(preds, [planes])], cfg, _default_device(device))
    _run_lists(session, [[(lambda: preds, planes, True, rng or _global_random, lambda: None)]], cfg, stats)
    return _write_back(preds, planes, cfg, 'trans')


def optimize_planes_3dc(preds, planes, frames=None, cfg=None, device=None, rng=None,
                        _session=None, stats=None):
    """Rotation tracks with 3-D clustering (reference utils/opt_utils.py:382-682)."""
    cfg, stats = cfg or OptConfig(), stats if stats is not None else Stats()
    session = _session or _Session([(preds, [planes])], cfg, _default_device(device))
    _run_lists(session, [[(lambda: preds, planes, False, rng or _global_random, lambda: None)]], cfg, stats)
    return _write_back(preds, planes, cfg, 'rot')


def optimize_planes_3d(preds, planes, cfg=None, device=None, rng=None, stats=None):
    """Legacy method '3d' (reference utils/opt_utils.py:112-379)."""
    cfg, stats = cfg or OptConfig(), stats if stats is not None else Stats()
    session = _Session([(preds, [planes])], cfg, _default_device(device))
    _run_lists(session, [[(lambda: preds, planes, False, rng or _global_random, lambda: None)]], cfg, stats,
               legacy=True)
    return _write_back(preds, planes, cfg, 'legacy')


def optimize_planes_average(preds, planes):
    """Method 'average' (reference utils/opt_utils.py:75-109); host only."""
    for plane in planes:
        std_axes = []
        for idx in plane['ids']:
            box_id = plane['ids'][idx]
            p_instance = preds[idx]
            pts = angle_offset_to_axis(p_instance.pred_rot_axis, p_instance.pred_boxes.get_centers())
            img_centers = torch.FloatTensor(np.array([[320, 240]]))
            std_axis = axis_to_angle_offset(pts.numpy().tolist(), img_centers)[:, :3]
            std_axes.append(std_axis[box_id:(box_id + 1)])
        plane['std_axis'] = torch.cat(std_axes).mean(axis=0)
    for idx, p_instance in enumerate(preds):
        for plane in planes:
            if idx in plane['ids']:
                p_instance.pred_rot_axis[plane['ids'][idx]] = plane['std_axis']
    return list(preds)


def _video_stages(preds, planes, cfg, rng, out):
    """The '3dc' method of one video as two stages: translation tracks on ``preds``, then rotation
    tracks on the translation stage's output (reference :968-970).  ``out[0]`` receives the result."""
    state = {"mid": None}

    def after_trans():
        state["mid"] = _write_back(preds, planes['trans'], cfg, 'trans')

    def after_rot():
        out[0] = _write_back(state["mid"], planes['rot'], cfg, 'rot')

    return [(lambda: preds, planes['trans'], True, rng, after_trans),
            (lambda: state["mid"], planes['rot'], False, rng, after_rot)]


def optimize_planes(preds, planes, method, frames=None, cfg=None, device=None, stats=None):
    """Reference dispatcher (utils/opt_utils.py:962-974).  ``planes`` is the dict
    ``track_planes`` returns for '3dc', a list of tracks for 'average' / '3d'."""
    if method == 'average':
        return optimize_planes_average(preds, planes)
    elif method == '3d':
        return optimize_planes_3d(preds, planes, cfg=cfg, device=device, stats=stats)
    elif method == '3dc':
        cfg = cfg or OptConfig()
        stats = stats if stats is not None else Stats()
        session = _Session([(preds, [planes['trans'], planes['rot']])], cfg, _default_device(device))
        stats.h2d_bytes += session.h2d_bytes
        out = [None]
        _run_lists(session, [_video_stages(preds, planes, cfg, _global_random, out)], cfg, stats)
        return out[0]
    else:
        raise NotImplementedError


def optimize_videos(videos, seeds, cfg=None, device=None, stats=None):
    """Batched '3dc' over independent videos: ``videos`` is a list of
    ``(preds, planes)``; video i draws its source frames from
    ``random.Random(seeds[i])`` (the reference seeds one process per video,
    tools/inference.py:172), so the result of every video equals
    ``random.seed(seeds[i]); optimize_planes(preds, planes, '3dc')``.  ``planes`` may be None: the video is
    then tracked here (``track_planes``) and ``videos[i]`` becomes ``(preds, planes)``.  All videos share one
    device session; their cluster phases are answered from one all-sources pass (few videos) or
    advance in lock-step, one job per video per device pass (many videos)."""
    cfg = cfg or OptConfig()
    stats = stats if stats is not None else Stats()
    device = _default_device(device)
    outs = [[None] for _ in videos]
    dense = all(_has(f, 'pred_masks') for p, _ in videos for f in p[:1])
    # ``(preds, None)``: the video is tracked here (``track_planes``) — in the pipelined schedule below when its
    # turn to be uploaded comes, i.e. behind the transfers of the videos before it instead of in front of all
    # of them; ``videos[i]`` is replaced by ``(preds, planes)``
    if not isinstance(videos, list):
        videos = list(videos)
    lazy = [pl is None for _, pl in videos]
    mode = os.environ.get("A3D_SCHEDULE") or cfg.schedule
    if not (videos and dense and any(lazy) and mode in ("table", "auto")):
        for v, (p, pl) in enumerate(videos):
            if pl is None:
                videos[v] = (p, track_planes(p, cfg))
        lazy = [False] * len(videos)

    def tables_for(v):
        p, pl = videos[v]
        return _use_tables([(v, pl['trans'], True), (v, pl['rot'], False)], cfg)
    if videos and dense and all(lazy[v] or tables_for(v) for v in range(len(videos))):
        # all-sources schedule, one session per video, software-pipelined: while video v is optimised
        # (table pass, host replay, final pass, write-back), the helper thread of session v+1 uploads and
        # packs the next video's masks on its own stream
        # ... and `pipeline_workers` videos are optimised at a time, each by its own thread on its own stream
        # with its own pass buffers: most of a video's time on the host is spent inside torch / CUDA calls
        # that release the interpreter lock (waiting for the table pass, float64 array arithmetic, copies).
        n_workers = max(1, min(int(os.environ.get("A3D_PIPELINE_WORKERS") or cfg.pipeline_workers), len(videos)))
        wss = [(engine.Workspace(device), engine.Staging(device)) for _ in range(n_workers)]
        ahead = n_workers + 1                       # sessions opened (uploads / preparation queued) ahead, in video order
        sessions, next_open, open_lock = {}, [0], threading.Lock()

        def open_upto(last):
            with open_lock:                         # in order: the upload and preparation queues are FIFO
                while next_open[0] <= min(last, len(videos) - 1):
                    v = next_open[0]
                    p, pl = videos[v]
                    if pl is None:
                        pl = track_planes(p, cfg)
                        videos[v] = (p, pl)
                    ws, staging = wss[v % n_workers]
                    sess = _Session([(p, [pl['trans'], pl['rot']])], cfg, device, ws=ws, staging=staging)
                    lists = [(0, planes, tr) for planes, tr in ((pl['trans'], True), (pl['rot'], False)) if planes]
                    if lists and sess.n_masks:
                        sess.prefetch_tables(lists)   # geometry + candidate transforms of all sources, off the workers
                    sessions[v] = sess
                    next_open[0] += 1

        def work(w, stream, wstats):
            torch.cuda.set_device(device)
            with torch.cuda.stream(stream):
                def start(v):
                    """Session of video v with its table passes enqueued (device work for the time the host
                    spends on the video before it)."""
                    open_upto(v + ahead - 1)
                    with open_lock:
                        session = sessions.pop(v)
                    p, pl = videos[v]
                    wstats.h2d_bytes += session.h2d_bytes
                    stages = [_video_stages(p, pl, cfg, _global_random.Random(seeds[v]), outs[v])]
                    lists = _table_lists(stages)
                    launched = session.launch_tables(lists, wstats) if lists and session.n_masks else None
                    return session, stages, launched
                mine = list(range(w, len(videos), n_workers))
                nxt = start(mine[0]) if mine else None
                for i, v in enumerate(mine):
                    session, stages, launched = nxt
                    nxt = start(mine[i + 1]) if i + 1 < len(mine) else None
                    _run_lists(session, stages, cfg, wstats, use_tables=True, launched=launched)

        open_upto(ahead - 1)
        main = torch.cuda.current_stream(device)
        if n_workers == 1:
            work(0, main, stats)
        else:
            streams = [torch.cuda.Stream(device=device) for _ in range(n_workers)]
            start = torch.cuda.Event()
            start.record(main)
            wstats = [Stats() for _ in range(n_workers)]
            errors = []

            def guarded(w):
                try:
                    streams[w].wait_event(start)
                    work(w, streams[w], wstats[w])
                except BaseException as e:             # re-raised below, on the caller's thread
                    errors.append(e)
            threads = [threading.Thread(target=guarded, args=(w,), name=f"a3d-video-{w}") for w in range(n_workers)]
            for t in threads:
                t.start()
            for t in threads:
                t.join()
            if errors:
                raise errors[0]
            for w, st in enumerate(streams):          # later work on the caller's stream sees the workers' results
                done = torch.cuda.Event()
                done.record(st)
                main.wait_event(done)
            for _, pl in videos:                      # the kept masks were allocated on a worker's stream
                for cat in ('trans', 'rot'):
                    for plane in pl[cat]:
                        rm = plane.get('reg_masks')
                        if isinstance(rm, RegMasks) and rm.packed is not None and rm.packed.is_cuda:
                            rm.packed.record_stream(main)
            for ws_ in wstats:
                for f in ("units_visited", "units_computed", "passes", "jobs", "h2d_bytes", "d2h_bytes"):
                    setattr(stats, f, getattr(stats, f) + getattr(ws_, f))
                stats.schedule = ws_.schedule or stats.schedule
        return [o[0] for o in outs]
    for v, (p, pl) in enumerate(videos):          # (untracked entries next to videos too big for the table schedule)
        if pl is None:
            videos[v] = (p, track_planes(p, cfg))
    session = _Session([(p, [pl['trans'], pl['rot']]) for p, pl in videos], cfg, device)
    stats.h2d_bytes += session.h2d_bytes
    _run_lists(session, [_video_stages(p, pl, cfg, _global_random.Random(s), o)
                         for (p, pl), s, o in zip(videos, seeds, outs)], cfg, stats)
    return [o[0] for o in outs]
