"""numpy restatement of a3d_plane_maps' output, bit for bit as include/a3d.h defines it: the oracle of the plane-map
tests.  Every float64 operation is a separate elementwise numpy operation in the header's order (numpy neither
fuses nor reorders them), z is rounded once to fp32, and a layer replaces the running best only when its z is
strictly smaller (ties keep the earlier layer)."""
import numpy as np


def rays(kinv, H: int, W: int):
    """(rx, ry, rz) float64 (H, W) of every pixel: the sparse form when kinv has the [[a,0,b],[0,c,d],[0,0,1]]
    pattern, the general one otherwise (the same values wherever both apply)."""
    k = np.asarray(kinv, dtype=np.float64).reshape(9)
    y, x = np.mgrid[0:H, 0:W].astype(np.float64)
    if k[1] == 0.0 and k[3] == 0.0 and k[6] == 0.0 and k[7] == 0.0 and k[8] == 1.0:
        return k[0] * x + k[2], k[4] * y + k[5], np.ones((H, W))
    return ((k[0] * x + k[1] * y) + k[2], (k[3] * x + k[4] * y) + k[5], (k[6] * x + k[7] * y) + k[8])


def plane_z(ray, normal, offset) -> np.ndarray:
    """fp32 z of every pixel's ray on the plane normal . X = offset (fp32 inputs widened to float64)."""
    rx, ry, rz = ray
    n = np.asarray(normal, dtype=np.float32).astype(np.float64)
    off = np.float64(np.float32(offset))
    with np.errstate(all="ignore"):
        dot = (n[0] * rx + n[1] * ry) + n[2] * rz
        return ((off / dot) * rz).astype(np.float32)


def plane_maps(kinv, masks, layers, layer_begin, bg_rgb=(0, 0, 0)):
    """(depth (T, H, W) fp32, rgb (T, H, W, 3) uint8).  ``masks`` (n, H, W) of the pool (nonzero = set)."""
    masks = np.asarray(masks) != 0
    H, W = masks.shape[-2:]
    ray = rays(kinv, H, W)
    T = len(layer_begin) - 1
    depth = np.zeros((T, H, W), np.float32)
    rgb = np.empty((T, H, W, 3), np.uint8)
    for f in range(T):
        best = np.full((H, W), np.inf, np.float32)
        col = np.empty((H, W, 3), np.uint8)
        col[:] = np.asarray(bg_rgb, np.uint8)
        for L in layers[layer_begin[f]:layer_begin[f + 1]]:
            m = int(L["mask"])
            if not 0 <= m < len(masks):
                continue
            z = plane_z(ray, L["normal"], L["offset"])
            with np.errstate(invalid="ignore"):
                win = masks[m] & (z > 0) & np.isfinite(z) & (z < best)
            best[win] = z[win]
            col[win] = L["rgb"]
        depth[f] = np.where(np.isfinite(best), best, np.float32(0))
        rgb[f] = col
    return depth, rgb
