"""ctypes binding of the C ABI in include/a3d.h (csrc/liba3d.so).

There is NO fallback: if the shared library is missing or a call fails, this
module raises.  Build the library with ``python -c "import __graft_entry__ as g;
g.build()"`` (or ``python -m articulation3d_b200.build``).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# A3D_LIB: a differently built copy of the same library (debug counters, tools/filter_stats.py)
LIB_PATH = os.environ.get("A3D_LIB") or os.path.join(_HERE, "csrc", "liba3d.so")

A3D_F32, A3D_U8 = 0, 1
OUT_FULL, OUT_BBOX_ROWS = 0, 1      # A3D_OUT_*: what a3d_project / a3d_pass write of every projected mask
MODE_SEQ, MODE_COMPOSED, MODE_TRANSLATE = 0, 1, 2
PCD_PLANES = 5          # A3D_PCD_PLANES: floats of point-cloud workspace per point
HOM_FLOATS = 12         # A3D_HOM_FLOATS: floats of homography workspace per candidate


class Camera(C.Structure):
    """a3d_camera_t"""
    _fields_ = [("kinv", C.c_double * 9), ("f", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("H", C.c_int32), ("W", C.c_int32)]


# a3d_job_t as a numpy structured dtype (72 bytes, C layout)
JOB_DTYPE = np.dtype([
    ("src_mask", "<i4"), ("mode", "<i4"), ("cand_begin", "<i4"), ("n_cand", "<i4"),
    ("tgt_begin", "<i4"), ("n_tgt", "<i4"),
    ("normal", "<f4", (3,)), ("offset", "<f4"),
    ("pivot", "<f4", (3,)), ("pcd_cap", "<i4"),
    ("tab_begin", "<i8"), ("pcd_begin", "<i8"),
], align=True)
assert JOB_DTYPE.itemsize == 72, JOB_DTYPE.itemsize

# a3d_layer_t / a3d_segment_t (a3d_render) as numpy structured dtypes, C layout
LAYER_FILL, LAYER_OUTLINE = 0, 1
LAYER_DTYPE = np.dtype([("mask", "<i4"), ("kind", "<i4"), ("rgba", "u1", (4,))])
SEGMENT_DTYPE = np.dtype([("x0", "<i4"), ("y0", "<i4"), ("x1", "<i4"), ("y1", "<i4"), ("radius", "<i4"),
                          ("rgb", "u1", (3,)), ("pad", "u1")])
assert LAYER_DTYPE.itemsize == 12 and SEGMENT_DTYPE.itemsize == 24
RENDER_MAX_SIDE = 16384      # A3D_RENDER_MAX_SIDE
RENDER_MAX_COORD = 1 << 14   # |segment coordinate| limit of a3d_render
RENDER_MAX_RADIUS = 256

# a3d_plane_layer_t (a3d_plane_maps) as a numpy structured dtype, C layout
PLANE_LAYER_DTYPE = np.dtype([("mask", "<i4"), ("normal", "<f4", (3,)), ("offset", "<f4"), ("rgb", "u1", (3,)),
                              ("pad", "u1")])
assert PLANE_LAYER_DTYPE.itemsize == 24

# every symbol include/a3d.h declares
EXPORTS = (
    "a3d_version", "a3d_last_error_string", "a3d_pitch_words", "a3d_project_max_tile",
    "a3d_pack_masks", "a3d_mask_meta", "a3d_project", "a3d_score", "a3d_pass", "a3d_emit_masks",
    "a3d_rle_to_bits", "a3d_plane_offsets", "a3d_plan_tiles", "a3d_host_quat_to_xform", "a3d_fetch_host_block", "a3d_upload_masks", "a3d_host_rle_counts",
    "a3d_rle_count_runs", "a3d_bits_to_rle", "a3d_host_rle_strings", "a3d_render",
    "a3d_plane_maps",
)

_lib = None


class A3DError(RuntimeError):
    pass


def load():
    """dlopen liba3d.so and declare the prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise A3DError(
            f"{LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`. "
            "articulation3d_b200 has no CPU fallback for the hot path.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    lib.a3d_version.restype = C.c_int
    lib.a3d_version.argtypes = []
    lib.a3d_last_error_string.restype = C.c_char_p
    lib.a3d_last_error_string.argtypes = []
    lib.a3d_pitch_words.restype = C.c_int
    lib.a3d_pitch_words.argtypes = [i32]
    lib.a3d_project_max_tile.restype = C.c_int
    lib.a3d_project_max_tile.argtypes = [i32, i32]
    lib.a3d_pack_masks.restype = C.c_int
    lib.a3d_pack_masks.argtypes = [vp, i32, i64, i32, i32, f32, vp, vp, vp]
    lib.a3d_mask_meta.restype = C.c_int
    lib.a3d_mask_meta.argtypes = [vp, i64, i32, i32, vp, vp, vp]
    lib.a3d_project.restype = C.c_int
    lib.a3d_project.argtypes = [C.POINTER(Camera), vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, vp, i32, vp]
    lib.a3d_score.restype = C.c_int
    lib.a3d_score.argtypes = [i32, i32, vp, i32, i32, i32, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                              vp, vp, vp, vp, vp]
    lib.a3d_pass.restype = C.c_int
    lib.a3d_pass.argtypes = [C.POINTER(Camera), vp, i32, i32, i32, i32, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp,
                             vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    lib.a3d_plan_tiles.restype = C.c_int
    lib.a3d_plan_tiles.argtypes = [vp, i32, i32, i32, vp, i32, C.POINTER(C.c_int)]
    lib.a3d_host_quat_to_xform.restype = C.c_int
    lib.a3d_host_quat_to_xform.argtypes = [vp, vp, i64, vp]
    lib.a3d_fetch_host_block.restype = C.c_int
    lib.a3d_fetch_host_block.argtypes = [vp, vp, i64, vp]
    lib.a3d_host_rle_counts.restype = C.c_int64
    lib.a3d_host_rle_counts.argtypes = [vp, vp, i64, vp, i64, vp, vp]
    lib.a3d_host_rle_strings.restype = C.c_int64
    lib.a3d_host_rle_strings.argtypes = [vp, vp, i64, vp, i64, vp]
    lib.a3d_upload_masks.restype = C.c_int
    lib.a3d_upload_masks.argtypes = [vp, vp, i32, i32, i32, i32, f32, vp, i64, vp, vp, i32, vp]
    lib.a3d_emit_masks.restype = C.c_int
    lib.a3d_emit_masks.argtypes = [vp, vp, i64, i32, i32, i32, vp, vp]
    lib.a3d_rle_to_bits.restype = C.c_int
    lib.a3d_rle_to_bits.argtypes = [vp, vp, i64, i32, i32, vp, vp]
    lib.a3d_rle_count_runs.restype = C.c_int
    lib.a3d_rle_count_runs.argtypes = [vp, vp, i64, i32, i32, vp, vp]
    lib.a3d_bits_to_rle.restype = C.c_int
    lib.a3d_bits_to_rle.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp]
    lib.a3d_plane_offsets.restype = C.c_int
    lib.a3d_plane_offsets.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, vp, i64, vp, vp, vp]
    lib.a3d_render.restype = C.c_int
    lib.a3d_render.argtypes = [vp, i64, i32, i32, i32, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    lib.a3d_plane_maps.restype = C.c_int
    lib.a3d_plane_maps.argtypes = [C.POINTER(Camera), i32, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc < 0:
        msg = load().a3d_last_error_string().decode("utf-8", "replace")
        raise A3DError(f"{what} failed ({rc}): {msg}")
    return rc


def pitch_words(W: int) -> int:
    """Pure-python twin of a3d_pitch_words (ceil(W/32) rounded up to 4 words)."""
    return (((W + 31) >> 5) + 3) & ~3
