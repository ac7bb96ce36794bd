"""Host-side scalar geometry of one source frame (a handful of flops per job).

What stays on the host, and why: the plane conversion, the integer axis
end-points, the two unprojected axis points, the unit axis direction and the
per-candidate rigid transforms are O(candidates) numbers per job and are built
in float64 with the same torch/numpy calls the reference makes, so they are
bit-identical by construction; the O(pixels x candidates) work runs on the
device (csrc/a3d.cu).  Reference call sites (utils/opt_utils.py):
:400-417 / :536-552 (rotation), :700-721 / :840-860 (translation),
:420-432, :553-574, :724-728 (transforms).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import torch
import torch.nn.functional as F

from .axis import angle_offset_to_axis, angle_offset_to_axis_rows
from .config import OptConfig


@dataclass
class SourceGeometry:
    normal: torch.Tensor        # (3,) fp32 unit normal, camera frame
    offset: torch.Tensor        # 0-dim fp32
    pts: torch.Tensor           # (n_boxes, 4) int64 axis end-points of every box of the frame
    axis3d: np.ndarray          # (2, 3) float64 unprojected end-points of this box's axis
    dir_vec: np.ndarray         # (3,) float64 unit axis direction
    pivot: np.ndarray           # (3,) fp32  = Translate(axis3d[0]) as pytorch3d stores it


def unproject_points(verts_xy, normal: torch.Tensor, offset: torch.Tensor, cfg: OptConfig) -> np.ndarray:
    """Ray/plane intersection of a few pixels in float64 (utils/vis.py:86-102),
    products and sums separately rounded, left to right — the same order the
    device kernel uses for the mask pixels."""
    K = cfg.K_inv()
    v = np.asarray(verts_xy, dtype=np.float64).reshape(-1, 2)
    x, y = v[:, 0], v[:, 1]
    n = normal.detach().cpu().numpy().astype(np.float32).astype(np.float64)
    off = np.float64(np.float32(float(offset)))
    with np.errstate(all="ignore"):
        rx = (K[0, 0] * x + K[0, 1] * y) + K[0, 2]
        ry = (K[1, 0] * x + K[1, 1] * y) + K[1, 2]
        rz = (K[2, 0] * x + K[2, 1] * y) + K[2, 2]
        depth = off / ((n[0] * rx + n[1] * ry) + n[2] * rz)
        return np.stack([depth * rx, depth * ry, depth * rz], axis=1)


def source_geometry(p_instance, box_id: int, cfg: OptConfig, translation: bool,
                    all_boxes: bool = False) -> SourceGeometry:
    """``pts`` holds the integer axis end-points; the reference computes them for every box
    of the frame and uses row ``box_id`` (all rows only in the legacy method's ``std_axis``),
    so by default only that row is computed (the others are zero)."""
    plane = p_instance.pred_planes[box_id:(box_id + 1)].clone()
    plane[:, [1, 2]] = plane[:, [2, 1]]            # [a, b, c] -> [a, -c, b]
    plane[:, 1] = -plane[:, 1]
    normal = F.normalize(plane, p=2)[0]
    offset = torch.norm(plane, p=2)
    centers = p_instance.pred_boxes.get_centers()
    if translation:
        axis = p_instance.pred_tran_axis
        axis = torch.cat((axis, torch.zeros(len(axis), 1)), 1)     # offset column = 0
    else:
        axis = p_instance.pred_rot_axis
    if all_boxes:
        pts = angle_offset_to_axis(axis, centers, H=cfg.height, W=cfg.width)
    else:
        pts = torch.zeros(len(axis), 4, dtype=torch.int64)
        pts[box_id] = angle_offset_to_axis(axis[box_id:box_id + 1], centers[box_id:box_id + 1],
                                           H=cfg.height, W=cfg.width)[0]
    axis3d = unproject_points(pts[box_id].reshape(-1, 2).numpy(), normal, offset, cfg)
    with np.errstate(all="ignore"):
        d = axis3d[1] - axis3d[0]
        d = d / np.linalg.norm(d)
    return SourceGeometry(normal, offset, pts, axis3d, d, axis3d[0].astype(np.float32))


@dataclass
class SourceGeometryRows:
    """``SourceGeometry`` of many independent (frame, box) sources, as numpy arrays."""
    normal: np.ndarray          # (n,3) fp32
    offset: np.ndarray          # (n,)  fp32
    pts: np.ndarray             # (n,4) int64 axis end-points of each source's own box
    axis3d: np.ndarray          # (n,2,3) float64
    dir_vec: np.ndarray         # (n,3) float64
    pivot: np.ndarray           # (n,3) fp32

    def __len__(self):
        return len(self.offset)

    def row(self, i: int, box_id: int, n_boxes: int) -> SourceGeometry:
        """Row ``i`` as the per-source record (``pts`` holds the row of ``box_id`` only)."""
        pts = torch.zeros(n_boxes, 4, dtype=torch.int64)
        pts[box_id] = torch.from_numpy(self.pts[i])
        return SourceGeometry(torch.from_numpy(self.normal[i].copy()), torch.tensor(self.offset[i]), pts,
                              self.axis3d[i], self.dir_vec[i], self.pivot[i])


def concat_rows(parts) -> SourceGeometryRows:
    if len(parts) == 1:
        return parts[0]
    return SourceGeometryRows(*(np.concatenate([getattr(p, f) for p in parts])
                                for f in ("normal", "offset", "pts", "axis3d", "dir_vec", "pivot")))


def source_geometry_rows(planes: torch.Tensor, axis: torch.Tensor, centers: torch.Tensor,
                         cfg: OptConfig) -> SourceGeometryRows:
    """``source_geometry`` for n independent sources in one set of array operations.

    planes (n,3) fp32 ``pred_planes`` rows; axis (n,3) fp32 ``[sin, cos, offset]`` rows
    (``pred_rot_axis``, or ``pred_tran_axis`` with a zero offset column); centers (n,2) fp32 box
    centres.  Every step is the per-source function's operation applied row-wise (row-wise torch
    norms, elementwise numpy fp32 / fp64), except the length of the axis direction, which stays
    one ``np.linalg.norm`` call per source: its BLAS dot product rounds differently from any
    array reduction.  tests/test_host_logic.py checks bit equality with ``source_geometry``."""
    plane = planes.detach().cpu().to(torch.float32).clone().reshape(-1, 3)
    plane[:, [1, 2]] = plane[:, [2, 1]]            # [a, b, c] -> [a, -c, b]
    plane[:, 1] = -plane[:, 1]
    normal = F.normalize(plane, p=2).numpy()
    offset = torch.norm(plane, p=2, dim=1).numpy()
    pts = angle_offset_to_axis_rows(axis.detach().cpu().numpy(), centers.detach().cpu().numpy(),
                                    H=cfg.height, W=cfg.width)
    n = len(offset)
    K = cfg.K_inv()
    nn = normal.astype(np.float64)
    off = offset.astype(np.float64)
    axis3d = np.empty((n, 2, 3), dtype=np.float64)
    with np.errstate(all="ignore"):
        for e in range(2):
            x = pts[:, 2 * e].astype(np.float64)
            y = pts[:, 2 * e + 1].astype(np.float64)
            rx = (K[0, 0] * x + K[0, 1] * y) + K[0, 2]
            ry = (K[1, 0] * x + K[1, 1] * y) + K[1, 2]
            rz = (K[2, 0] * x + K[2, 1] * y) + K[2, 2]
            depth = off / ((nn[:, 0] * rx + nn[:, 1] * ry) + nn[:, 2] * rz)
            axis3d[:, e, 0], axis3d[:, e, 1], axis3d[:, e, 2] = depth * rx, depth * ry, depth * rz
        d = axis3d[:, 1] - axis3d[:, 0]
        # np.linalg.norm of a 1-D vector is sqrt(v.dot(v)); the dot product stays the per-source BLAS call
        length = np.sqrt(np.fromiter((v.dot(v) for v in d), dtype=np.float64, count=n))
        d = d / length[:, None]
    return SourceGeometryRows(normal, offset, pts, axis3d, d, axis3d[:, 0].astype(np.float32))


def _axis_angle_to_matrix(axis_angle: torch.Tensor) -> torch.Tensor:
    """Rotation matrices of axis-angle vectors via unit quaternions, in the input
    dtype (float64 here) — the construction pytorch3d's ``axis_angle_to_matrix``
    documents: q = [cos(t/2), v sin(t/2)/t] (Taylor 1/2 - t^2/48 for |t| < 1e-6),
    R from two_s = 2/|q|^2, e.g. R00 = 1 - two_s (jj + kk), R01 = two_s (ij - kr).
    Returns (..., 9) row-major entries.  All steps are torch ops (its sin/cos and its reductions: numpy's
    float64 sin differs in the last ulp); the nine entries are evaluated on contiguous component
    planes — per entry the same multiplications and additions in the same order as the oracle's form
    (tests/test_host_logic.py compares the bits)."""
    t = torch.norm(axis_angle, p=2, dim=-1, keepdim=True)
    half = t * 0.5
    k = torch.sin(half) / t
    small = t.abs() < 1e-6
    if bool(small.any()):
        k = torch.where(small, 0.5 - (t * t) / 48, k)
    q = torch.cat([torch.cos(half), axis_angle * k], dim=-1)
    two_s = 2.0 / (q * q).sum(-1)
    qt = q.movedim(-1, 0).contiguous()
    r, i, j, kk = qt[0], qt[1], qt[2], qt[3]
    ii, jj, k2 = i * i, j * j, kk * kk
    ij, ik, jk = i * j, i * kk, j * kk
    ir, jr, kr = i * r, j * r, kk * r
    return torch.stack((1 - two_s * (jj + k2), two_s * (ij - kr), two_s * (ik + jr),
                        two_s * (ij + kr), 1 - two_s * (ii + k2), two_s * (jk - ir),
                        two_s * (ik - jr), two_s * (jk + ir), 1 - two_s * (ii + jj)), -1)


def _rotation_entries(grid, dir_vec) -> torch.Tensor:
    """(A,) grid x (..., 3) float64 axis -> (..., A, 9) float64 entries: fp32 angles times the float64
    axis, matrix in float64 (all torch: the form the tests compare with the oracle's)."""
    angles = torch.as_tensor(np.asarray(grid), dtype=torch.float32)[:, None]       # (A,1)
    d = torch.as_tensor(np.asarray(dir_vec, dtype=np.float64))
    return _axis_angle_to_matrix(angles * d[..., None, :])


def _rotation_xforms(grid, dir_vec) -> np.ndarray:
    """(A,) grid x (..., 3) float64 axis -> (..., A, 12) fp32 candidate rows [R row-major | 0 0 0].

    The same values as ``_rotation_entries(...).to(float32)``: norms, sin / cos, the quaternion and
    ``two_s`` are the same torch calls; the nine entries (products and sums of quaternion components, IEEE
    arithmetic in the order of ``_axis_angle_to_matrix``) are evaluated in one fused pass by the library's
    host helper instead of ~40 array operations (tests/test_host_logic.py compares the bits)."""
    from . import _lib
    angles = torch.as_tensor(np.asarray(grid), dtype=torch.float32)[:, None]       # (A,1)
    d = torch.as_tensor(np.asarray(dir_vec, dtype=np.float64))
    axis_angle = angles * d[..., None, :]
    t = torch.norm(axis_angle, p=2, dim=-1, keepdim=True)
    half = t * 0.5
    k = torch.sin(half) / t
    small = t.abs() < 1e-6
    if bool(small.any()):
        k = torch.where(small, 0.5 - (t * t) / 48, k)
    q = torch.cat([torch.cos(half), axis_angle * k], dim=-1).contiguous()
    two_s = (2.0 / (q * q).sum(-1)).contiguous()
    out = np.zeros(tuple(q.shape[:-1]) + (12,), dtype=np.float32)
    _lib.check(_lib.load().a3d_host_quat_to_xform(q.data_ptr(), two_s.data_ptr(), two_s.numel(), out.ctypes.data),
               "a3d_host_quat_to_xform")
    return out


def rotation_matrices(grid, dir_vec) -> np.ndarray:
    """(A,) grid x (..., 3) float64 axis -> (..., A, 3, 3) fp32 (what ``Rotate`` keeps)."""
    x = _rotation_xforms(grid, dir_vec)
    return np.ascontiguousarray(x[..., :9]).reshape(x.shape[:-1] + (3, 3))


def xforms_seq(R: np.ndarray) -> np.ndarray:
    """Cluster phase: R only (the pivot travels in the job record).  (..., A, 12) fp32."""
    out = np.zeros(R.shape[:-2] + (12,), dtype=np.float32)
    out[..., :9] = R.reshape(R.shape[:-2] + (9,))
    return out


def xforms_seq_from_dirs(grid, dir_vec) -> np.ndarray:
    """``xforms_seq(rotation_matrices(grid, dir_vec))`` without the intermediate copies."""
    return _rotation_xforms(grid, dir_vec)


def xforms_composed(R: np.ndarray, pivot: np.ndarray) -> np.ndarray:
    """Final phase: one composed fp32 matrix (M_t3 M_R) M_t1; its last row is
    ((-a0 R0j + -a1 R1j) + -a2 R2j) + a_j, every step rounded to fp32."""
    a = np.asarray(pivot, dtype=np.float32)
    with np.errstate(all="ignore"):
        na = -a
        t = (na[..., None, 0, None] * R[..., 0, :] + na[..., None, 1, None] * R[..., 1, :]) \
            + na[..., None, 2, None] * R[..., 2, :]
        t = (t + a[..., None, :]).astype(np.float32)
    out = np.empty(R.shape[:-2] + (12,), dtype=np.float32)
    out[..., :9] = R.reshape(R.shape[:-2] + (9,))
    out[..., 9:] = t
    return out


def xforms_translate(grid, dir_vec) -> np.ndarray:
    """Translation candidates: fp32 offsets x float64 direction, stored fp32."""
    g = torch.as_tensor(grid, dtype=torch.float32)[:, None]
    d = torch.as_tensor(np.asarray(dir_vec, dtype=np.float64))
    v = (g * d[..., None, :]).to(torch.float32).numpy()
    out = np.zeros(v.shape[:-1] + (12,), dtype=np.float32)
    out[..., 0] = out[..., 4] = out[..., 8] = 1.0
    out[..., 9:] = v
    return out


def transform_normals(normal: torch.Tensor, R: np.ndarray) -> torch.Tensor:
    """Normals under the composed transform: n (M^T)^-1 over the 3x3 block (fp32)."""
    m = torch.from_numpy(np.ascontiguousarray(R))
    n = normal.reshape(1, 1, 3).expand(len(m), -1, -1)
    return n.bmm(m.transpose(1, 2).inverse())[:, 0]


def registered_planes(normal: torch.Tensor, offset, xform_rows: np.ndarray, mode: int, pivot, cand,
                      normals: torch.Tensor | None = None) -> np.ndarray:
    """Planes of the source mask moved by candidates ``cand`` of a job: (len(cand), 4) fp32 rows [n', d'] with
    n' . p' = d' for every point p' = p R + t of the moved plane n . p = offset (camera frame of get_pcd).

    ``xform_rows`` (A, 12) are the job's candidate rows (R row-major, t).  n' = n (R^T)^-1 is
    ``transform_normals`` (the fp32 value ``reg_normals`` is built from; ``normals`` may pass it in when already
    computed for all A rows); R = I for ``MODE_TRANSLATE`` (n' = n); for ``MODE_SEQ`` t = a - a R with a the fp32
    ``pivot``, in float64.  d' = fp32 of the float64 d + n'.t, exact for any invertible R:
    n . p = d  <=>  n' . p' = d + n' . t."""
    from . import _lib
    rows = np.asarray(xform_rows, dtype=np.float32).reshape(-1, 12)
    cand = np.asarray(cand, dtype=np.int64).reshape(-1)
    R = rows[:, :9].reshape(-1, 3, 3)
    if mode == _lib.MODE_TRANSLATE:
        n_sel = np.broadcast_to(normal.detach().cpu().numpy().astype(np.float32).reshape(1, 3), (len(cand), 3))
    else:
        if normals is None:
            normals = transform_normals(normal, R)
        n_sel = normals.numpy()[cand]
    Rs = R[cand].astype(np.float64)
    if mode == _lib.MODE_SEQ:
        a = np.asarray(pivot, dtype=np.float32).astype(np.float64)
        t = a[None, :] - ((a[0] * Rs[:, 0, :] + a[1] * Rs[:, 1, :]) + a[2] * Rs[:, 2, :])
    else:
        t = rows[cand, 9:].astype(np.float64)
    n64 = n_sel.astype(np.float64)
    with np.errstate(all="ignore"):
        d = np.float64(np.float32(float(offset))) + ((n64[:, 0] * t[:, 0] + n64[:, 1] * t[:, 1]) + n64[:, 2] * t[:, 2])
    out = np.empty((len(cand), 4), dtype=np.float32)
    out[:, :3] = n_sel
    out[:, 3] = d.astype(np.float32)
    return out
