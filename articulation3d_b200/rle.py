"""COCO run-length masks without pycocotools (SURVEY.md §8f row f2).

The reference's prediction records carry instance masks as COCO RLE
(``{'size': [h, w], 'counts': <compressed string | list>}``, written by
evaluation/arti_evaluation.py:153-180 through detectron2's
``instances_to_coco_json``; decoded with ``pycocotools.mask.decode`` in
utils/arti_vis.py:182 and :135).  pycocotools is a C extension that is not
a dependency here, so the codec is restated from the published format
[3P-unverified against the C source, pinned by round-trip tests]:

* runs alternate 0s and 1s, starting with 0s, over the mask in COLUMN-major
  (Fortran) order;
* the compressed string stores each count as a little-endian base-32 varint, 5
  payload bits per character plus a continuation bit (0x20), offset by 48 into
  printable ASCII, sign-extended from bit 4 of the last group; counts beyond the
  second are stored as differences to the count two places earlier.

``counts_to_bits`` turns run lengths into the bit-packed row-major layout of the
mask pool on the device (csrc/a3d.cu: k_rle_to_bits), so fp32 masks never exist.
"""
from __future__ import annotations

import numpy as np


def string_to_counts(s) -> np.ndarray:
    """Compressed COCO RLE string -> run lengths (uint32)."""
    if isinstance(s, str):
        s = s.encode("ascii")
    counts = []
    p, n = 0, len(s)
    while p < n:
        x, k, more = 0, 0, True
        while more:
            c = s[p] - 48
            x |= (c & 0x1F) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)
        if len(counts) > 2:
            x += counts[-2]
        counts.append(x)
    return np.asarray(counts, dtype=np.int64).astype(np.uint32)


def strings_to_counts(strings):
    """Many compressed strings at once, decoded by the library's host helper (``a3d_host_rle_counts``: the
    per-string Python loop above costs 40 us per simple mask).  Returns (flat uint32 counts, int64 begin[n+1],
    int64 run sums[n])."""
    import ctypes as C
    from . import _lib
    lib = _lib.load()
    bs = [x.encode("ascii") if isinstance(x, str) else bytes(x) for x in strings]
    n = len(bs)
    begin = np.zeros(n + 1, dtype=np.int64)
    if n:
        np.cumsum([len(b) for b in bs], out=begin[1:])
    blob = b"".join(bs)
    chars = np.frombuffer(blob, dtype=np.uint8) if blob else np.zeros(1, np.uint8)
    cbeg = np.zeros(n + 1, dtype=np.int64)
    sums = np.zeros(max(n, 1), dtype=np.int64)
    # every count takes at least one character
    counts = np.empty(max(len(blob), 1), dtype=np.uint32)
    total = _lib.check(lib.a3d_host_rle_counts(chars.ctypes.data, begin.ctypes.data, n, counts.ctypes.data, len(counts),
                                               cbeg.ctypes.data, sums.ctypes.data), "a3d_host_rle_counts")
    return counts[:total], cbeg, sums[:n]


def counts_to_string(counts) -> bytes:
    """Run lengths -> compressed COCO RLE string."""
    counts = [int(c) for c in counts]
    out = bytearray()
    for i, x in enumerate(counts):
        if i > 2:
            x -= counts[i - 2]
        more = True
        while more:
            c = x & 0x1F
            x >>= 5
            more = (x != -1) if (c & 0x10) else (x != 0)
            if more:
                c |= 0x20
            out.append(c + 48)
    return bytes(out)


def encode(mask: np.ndarray) -> dict:
    """(H, W) binary mask -> {'size': [H, W], 'counts': bytes} (column-major runs)."""
    m = np.asarray(mask).astype(bool)
    h, w = m.shape
    flat = m.T.reshape(-1)                       # column-major order
    if flat.size == 0:
        return {"size": [h, w], "counts": b""}
    change = np.flatnonzero(flat[1:] != flat[:-1]) + 1
    bounds = np.concatenate(([0], change, [flat.size]))
    runs = np.diff(bounds).tolist()
    if flat[0]:
        runs = [0] + runs                        # runs always start with zeros
    return {"size": [h, w], "counts": counts_to_string(runs)}


def counts_to_strings(counts, begin) -> list:
    """Run lengths of many masks (flat uint32 ``counts``, int64 ``begin[n+1]``) -> their compressed strings, written
    by the library's host helper (``a3d_host_rle_strings``, byte for byte ``counts_to_string``)."""
    from . import _lib
    lib = _lib.load()
    counts = np.ascontiguousarray(counts, dtype=np.uint32)
    begin = np.ascontiguousarray(begin, dtype=np.int64)
    n = len(begin) - 1
    cap = 7 * max(len(counts), 1)                 # a difference of two uint32 counts takes at most 7 characters
    chars = np.empty(cap, dtype=np.uint8)
    cbeg = np.zeros(n + 1, dtype=np.int64)
    _lib.check(lib.a3d_host_rle_strings(counts.ctypes.data, begin.ctypes.data, n, chars.ctypes.data, cap,
                                        cbeg.ctypes.data), "a3d_host_rle_strings")
    blob = chars.tobytes()
    return [blob[cbeg[i]:cbeg[i + 1]] for i in range(n)]


def bits_to_rles(bits, H: int, W: int, index=None) -> list:
    """Packed masks on the device ((n, H, pitch) int32, ``index`` as in ``engine.emit_masks``) -> COCO RLE dicts,
    encoded on the GPU (``engine.bits_to_rle``) with the strings written on the host."""
    from . import engine
    counts, begin = engine.bits_to_rle(bits, H, W, index)
    return [{"size": [H, W], "counts": s} for s in counts_to_strings(counts, begin)]


ENCODE_CHUNK = 256      # masks per host-to-device upload of encode_many (a 640x480 fp32 chunk is 315 MB)


def encode_many(masks, device=None) -> list:
    """``[encode(m) for m in masks]``, byte for byte, for an (n, H, W) fp32 / uint8 / bool stack of masks (numpy or
    torch, host or CUDA).  Without a device (``device=None`` and host masks) that is what it does.  Otherwise
    the masks are packed (``!= 0``, as ``encode`` tests them: NaN is set, -0.0 is not) and encoded on the GPU;
    host masks are uploaded ``ENCODE_CHUNK`` at a time, so the dense stack never sits on the device whole."""
    import torch
    from . import engine
    if isinstance(masks, np.ndarray):
        masks = torch.from_numpy(masks)
    if device is None and masks.is_cuda:
        device = masks.device
    n, H, W = masks.shape
    if device is None or n == 0 or H * W == 0:
        return [encode(m.numpy()) for m in masks.cpu()]
    device = torch.device(device)
    if device.type != "cuda":
        raise ValueError(f"encode_many encodes on a CUDA device, not {device}")
    pool = engine.PoolBuilder(n, H, W, device, with_nonzero=True)
    with torch.cuda.device(device):
        for lo in range(0, n, ENCODE_CHUNK):
            pool.append(masks[lo:lo + ENCODE_CHUNK].to(device))
    return bits_to_rles(pool.nz, H, W)


def rle_counts(rle: dict) -> np.ndarray:
    c = rle["counts"]
    if isinstance(c, (bytes, str)):
        return string_to_counts(c)
    return np.asarray(c, dtype=np.uint32)


def decode(rle: dict) -> np.ndarray:
    """RLE -> (H, W) uint8 mask (host reference implementation; the hot path uses
    ``engine.rle_to_pool`` instead)."""
    h, w = rle["size"]
    counts = rle_counts(rle).astype(np.int64)
    vals = np.zeros(len(counts), dtype=np.uint8)
    vals[1::2] = 1
    flat = np.repeat(vals, counts)
    if flat.size != h * w:
        raise ValueError(f"RLE covers {flat.size} pixels, mask is {h}x{w}")
    return flat.reshape(w, h).T.copy()
