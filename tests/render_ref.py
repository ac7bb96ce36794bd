"""numpy restatement of a3d_render's output, byte for byte as include/a3d.h defines it: the oracle of the render
tests and of tools/render_bench.py's host alternative."""
import numpy as np

from articulation3d_b200 import _lib


def outline(m: np.ndarray) -> np.ndarray:
    """Set pixels with at least one unset 4-neighbour; outside the frame counts as unset."""
    p = np.pad(np.asarray(m, bool), 1)
    inner = p[:-2, 1:-1] & p[2:, 1:-1] & p[1:-1, :-2] & p[1:-1, 2:]
    return p[1:-1, 1:-1] & ~inner


def segment_cover(H: int, W: int, x0: int, y0: int, x1: int, y1: int, r: int) -> np.ndarray:
    """Pixels whose squared distance to the closed segment is <= r^2, decided in int64 as the header states."""
    y, x = np.mgrid[0:H, 0:W].astype(np.int64)
    dx, dy = np.int64(x1) - x0, np.int64(y1) - y0
    qx, qy = x - x0, y - y0
    t, L, r2 = qx * dx + qy * dy, dx * dx + dy * dy, np.int64(r) * r
    ex, ey = x - x1, y - y1
    c = qx * dy - qy * dx
    return np.where(t <= 0, qx * qx + qy * qy <= r2, np.where(t >= L, ex * ex + ey * ey <= r2, c * c <= r2 * L))


def blend(c, o, a):
    c, o, a = (np.asarray(v, dtype=np.uint32) for v in (c, o, a))
    return ((c * a + o * (np.uint32(255) - a) + np.uint32(127)) // np.uint32(255)).astype(np.uint8)


def composite(background, masks, layers, layer_begin, segs, seg_begin) -> np.ndarray:
    """(T, H, W, 3) uint8.  ``masks`` (n, H, W) of the pool (nonzero = set); ``background`` (H, W, 3) or (T, H, W, 3)."""
    bg = np.asarray(background, dtype=np.uint8)
    H, W = bg.shape[-3], bg.shape[-2]
    masks = np.asarray(masks).reshape(-1, H, W) != 0
    T = len(layer_begin) - 1
    out = np.empty((T, H, W, 3), np.uint8)
    for f in range(T):
        img = (bg if bg.ndim == 3 else bg[f]).copy()
        for L in layers[layer_begin[f]:layer_begin[f + 1]]:
            m = int(L["mask"])
            if not 0 <= m < len(masks):
                continue
            cov = masks[m] if int(L["kind"]) == _lib.LAYER_FILL else outline(masks[m])
            img[cov] = blend(L["rgba"][:3][None, :], img[cov], L["rgba"][3])
        for S in segs[seg_begin[f]:seg_begin[f + 1]]:
            x0, y0, x1, y1, r = (int(S[k]) for k in ("x0", "y0", "x1", "y1", "radius"))
            # only the segment's box can be covered: decide the pixels of its part inside the frame
            bx0, bx1 = max(0, min(x0, x1) - r), min(W - 1, max(x0, x1) + r)
            by0, by1 = max(0, min(y0, y1) - r), min(H - 1, max(y0, y1) + r)
            if bx0 > bx1 or by0 > by1:
                continue
            cov = segment_cover(by1 - by0 + 1, bx1 - bx0 + 1, x0 - bx0, y0 - by0, x1 - bx0, y1 - by0, r)
            img[by0:by1 + 1, bx0:bx1 + 1][cov] = S["rgb"]
        out[f] = img
    return out
