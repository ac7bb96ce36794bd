"""``k_plane_offsets`` (``engine.plane_offsets``, ``a3d_plane_offsets``) against a float64 reference of the numerics
the kernel states: per mask pixel the fp32 chain X = r_x*d, Y = r_y*d, Z = r_z*d, t = (n0*X + n1*Y) + n2*Z with
every operation rounded on its own, the terms summed in fp64, the mean rounded once to fp32.

Counts are exact.  Offsets are bit-equal wherever the fp64 sum is exact in every order (``reference`` says when),
and within one fp32 ulp plus the fp64 summation bound elsewhere.  Depth, rays and normals on grids keep whole
frames in the exact regime while their fp32 products still round, so a float accumulator, a contracted product,
a skipped word column, a pixel or frame read outside the mask (NaN poison) or flushed denormals change bits."""
import math

import numpy as np
import pytest
import torch

from articulation3d_b200 import _lib, engine, rle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
A3D_OK, A3D_EINVAL, A3D_ELIMIT = 0, -1, -3          # include/a3d.h
NO_BIT = 1 << 20                                    # lowest-bit exponent of a zero term: larger than any real one


def _host_keeps_denormals():
    # torch.set_flush_denormal(True) also flushes numpy's float32 arithmetic, and the reference with it
    assert np.float32(1e-45) * np.float32(1) != 0, "the host flushes denormals: the fp32 reference would be wrong"


def _seg(ufunc, a, starts, counts, empty):
    """``ufunc`` over each instance's run of ``a`` (instance i owns a[starts[i]:starts[i] + counts[i]])."""
    out = np.full(len(counts), empty, dtype=np.result_type(a, type(empty)))
    ne = counts > 0
    if ne.any():
        out[ne] = ufunc.reduceat(a, starts[ne])
    return out


def reference(masks, inst_mask, normals, rays, depth=None, inst_frame=None):
    """Per instance: (offset fp32, count, bitwise, sum |t|).

    ``bitwise`` says the kernel must match ``offset`` bit for bit.  That holds when the result is not finite (NaN
    if a term is NaN or both infinities occur, else the infinity that occurs: every order of the fp64 sum gives
    that), and for finite terms when every order of the fp64 sum is exact or rounds once:
    * with 2^q the lowest set bit over the terms, every partial sum in any order is a multiple of 2^q of magnitude
      at most sum |t|; below 2^(53+q) it is a double, so the sum is exact (and equal to ``math.fsum``);
    * with at most two nonzero terms, whatever the order, the only inexact addition is the one of the two terms,
      rounded once to nearest: ``math.fsum`` of them.
    An exact zero sum is +0, as the kernel's accumulators start at +0 and x + (-x) = +0."""
    masks = np.asarray(masks, dtype=bool)
    inst_mask = np.asarray(inst_mask, dtype=np.int64)
    n = len(inst_mask)
    H, W = masks.shape[1:]
    pix = [np.flatnonzero(m) for m in masks.reshape(len(masks), -1)]
    counts = np.array([len(pix[m]) for m in inst_mask], dtype=np.int64)
    starts = np.concatenate(([0], np.cumsum(counts)[:-1])).astype(np.int64)
    flat = np.concatenate([pix[m] for m in inst_mask]) if n else np.zeros(0, np.int64)
    inst = np.repeat(np.arange(n), counts)
    r = np.asarray(rays, dtype=np.float32).reshape(3, H * W)
    nrm = np.asarray(normals, dtype=np.float32)
    if depth is None:
        d = np.float32(1.0)
    else:
        d = np.asarray(depth, dtype=np.float32).reshape(-1, H * W)[np.asarray(inst_frame)[inst], flat]
    with np.errstate(all="ignore"):
        X, Y, Z = r[0, flat] * d, r[1, flat] * d, r[2, flat] * d
        t = (nrm[inst, 0] * X + nrm[inst, 1] * Y) + nrm[inst, 2] * Z
    assert t.dtype == np.float32
    nan = _seg(np.logical_or, np.isnan(t), starts, counts, False)
    pinf = _seg(np.logical_or, t == np.inf, starts, counts, False)
    ninf = _seg(np.logical_or, t == -np.inf, starts, counts, False)
    tf = np.where(np.isfinite(t), t, 0).astype(np.float64)
    mant, ex = np.frexp(tf)
    m24 = np.abs(mant * 2.0 ** 24).astype(np.int64)          # every fp32 value has at most 24 significant bits
    low = np.where(m24 != 0, ex - 24 + np.frexp((m24 & -m24).astype(np.float64))[1] - 1, NO_BIT)
    q = _seg(np.minimum, low, starts, counts, NO_BIT)
    abs_sum = _seg(np.add, np.abs(tf), starts, counts, 0.0)
    nonzero = _seg(np.add, (tf != 0).astype(np.int64), starts, counts, 0)
    exact = (q == NO_BIT) | (abs_sum < np.ldexp(1.0, np.clip(53 + q, -1074, 1023).astype(np.int32)))
    bitwise = exact | (nonzero <= 2) | nan | pinf | ninf
    s = _seg(np.add, tf, starts, counts, 0.0)                 # exact, or one rounding, where bitwise
    for i in np.flatnonzero(~bitwise):
        s[i] = math.fsum(tf[starts[i]:starts[i] + counts[i]])
    s = s + 0.0                                               # -0 -> +0
    with np.errstate(all="ignore"):
        off = np.where(counts > 0, s / np.maximum(counts, 1), 0.0).astype(np.float32)
    off[pinf & ~ninf] = np.inf
    off[ninf & ~pinf] = -np.inf
    off[nan | (pinf & ninf)] = np.nan
    return off, counts, bitwise, abs_sum


def offset_tolerance(ref, got, abs_sum):
    """Bound on |got - ref| where the kernel's fp64 sum may round: one fp32 ulp (both results are the fp32
    rounding of means within the fp64 error of each other) plus 2^-52 sum |t| (recursive fp64 summation of c terms
    errs by at most (c - 1) 2^-53 sum |t|; the mean by 1/c of that, the double division by 2^-53 of the mean)."""
    ulp = np.maximum(np.spacing(np.abs(ref)), np.spacing(np.abs(got))).astype(np.float64)
    return ulp + 2.0 ** -52 * abs_sum


def assert_offsets(off, cnt, want, what=""):
    ref, counts, bitwise, abs_sum = want
    got = off.cpu().numpy() if torch.is_tensor(off) else np.asarray(off)
    c = cnt.cpu().numpy() if torch.is_tensor(cnt) else np.asarray(cnt)
    bad = np.flatnonzero(c != counts)
    assert bad.size == 0, f"{what} counts differ at {bad[:8].tolist()}: {c[bad[:8]].tolist()} != {counts[bad[:8]].tolist()}"
    nan = np.isnan(ref)
    bad = np.flatnonzero(np.isnan(got) != nan)
    assert bad.size == 0, f"{what} NaN differs at {bad[:8].tolist()}: {got[bad[:8]].tolist()} vs {ref[bad[:8]].tolist()}"
    bits = bitwise & ~nan
    bad = np.flatnonzero(bits & (got.view(np.int32) != ref.view(np.int32)))
    assert bad.size == 0, (f"{what} not bit-equal at {bad[:8].tolist()}: {got[bad[:8]].tolist()} "
                           f"!= {ref[bad[:8]].tolist()}")
    loose = ~bitwise & ~nan
    err = np.abs(got[loose].astype(np.float64) - ref[loose].astype(np.float64))
    tol = offset_tolerance(ref[loose], got[loose], abs_sum[loose])
    bad = np.flatnonzero(~(err <= tol))
    assert bad.size == 0, f"{what} off by {err[bad[:8]].tolist()} > {tol[bad[:8]].tolist()}"


def reference_planes(planes, masks, frame_of, rays, depth=None):
    """What ``adapter.override_depth*`` must return for input ``pred_plane`` rows ``planes`` (n, 3), instance masks
    (n, H, W) and depth frames ``frame_of``: (want (n, 3) fp32, tol (n, 3) float64).  The normal is the adapter's
    own torch expression on the CPU and the offset the float64 reference; a plane is normal * offset with the
    reference's swap, an empty mask keeps its plane.  Per component the bound is |n_i| times the offset's bound
    plus one ulp of the product, and 0 (bit-equal) where the offset is bit-equal."""
    p = planes.clone().float()
    p[:, [1, 2]] = p[:, [2, 1]]
    p[:, 1] = -p[:, 1]
    offset = torch.linalg.vector_norm(p, dim=1)
    normal = p / offset.clamp_min(1e-8)[:, None]
    ref, counts, bitwise, abs_sum = reference(masks, np.arange(len(p)), normal.numpy(), rays, depth, frame_of)
    tol_off = np.where(bitwise, 0.0, offset_tolerance(ref, np.nextafter(np.abs(ref), np.float32(np.inf)), abs_sum))
    want = torch.where(torch.from_numpy(counts > 0)[:, None], normal * torch.from_numpy(ref)[:, None], p)
    tol = normal.abs().numpy() * tol_off[:, None] + (tol_off > 0)[:, None] * np.spacing(np.abs(want.numpy()))
    for t in (want, tol):
        t[:, [1, 2]] = t[:, [2, 1]]
    want[:, 2] = -want[:, 2]
    assert torch.equal(want[counts == 0].view(torch.int32), planes[counts == 0].float().view(torch.int32))
    return want, tol


def assert_planes(got, want, what=""):
    want, tol = want
    err = (got.double() - want.double()).abs().numpy()
    bad = np.argwhere(~(err <= tol))
    assert bad.size == 0, f"{what} planes off at {bad[:4].tolist()}: {err[~(err <= tol)][:4]} > {tol[~(err <= tol)][:4]}"
    exact = tol == 0
    assert np.array_equal(got.view(torch.int32).numpy()[exact], want.view(torch.int32).numpy()[exact]), what


def _grid(rng, shape, lo, hi, step):
    """fp32 values on multiples of ``step`` in [lo, hi]."""
    return rng.randint(int(lo / step), int(hi / step) + 1, size=shape, dtype=np.int32).astype(np.float32) * np.float32(step)


def _normal_step(H, W):
    # terms are multiples of 2^-10 (rays) * 2^-8 (depth) * step and at most 3 * 2 * 4 = 24 in magnitude: a whole
    # 480x640 mask stays below 2^53 times the lowest bit with 2^-12, bigger frames need a coarser grid
    return 2.0 ** -12 if H * W <= 480 * 640 else 2.0 ** -6


def _pools(masks):
    """The packed pool of ``masks`` and, where the RLE decoder holds the frame in shared memory, the decoded
    pool of their COCO strings."""
    H, W = masks.shape[1:]
    packed = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    smem = torch.cuda.get_device_properties(DEV).shared_memory_per_block_optin
    if H * _lib.pitch_words(W) * 4 > smem - 8192:                  # a3d_rle_to_bits refuses these
        return packed, None
    return packed, engine.rle_to_pool([rle.encode(m) for m in masks], H, W, DEV)


def run_case(masks, inst_mask, normals, rays, depth=None, inst_frame=None, exact=True, what=""):
    """Offsets of both pools against the reference; with ``exact`` every instance must be in the bit-equal
    regime (a case built to be exact that is not fails instead of falling back to the tolerance)."""
    _host_keeps_denormals()
    want = reference(masks, inst_mask, normals, rays, depth, inst_frame)
    if exact:
        assert want[2].all(), f"{what}: instances {np.flatnonzero(~want[2])[:8].tolist()} are not exact sums"
    args = [torch.as_tensor(np.asarray(inst_mask, np.int32), device=DEV),
            torch.from_numpy(np.ascontiguousarray(normals, np.float32)).to(DEV),
            torch.from_numpy(np.ascontiguousarray(rays, np.float32)).to(DEV)]
    if depth is not None:
        args += [torch.from_numpy(np.ascontiguousarray(depth, np.float32)).to(DEV),
                 torch.as_tensor(np.asarray(inst_frame, np.int32), device=DEV)]
    packed, decoded = _pools(masks)
    off, cnt = engine.plane_offsets(packed, *args)
    assert_offsets(off, cnt, want, what)
    if decoded is not None:
        off2, cnt2 = engine.plane_offsets(decoded, *args)
        assert torch.equal(off2.view(torch.int32), off.view(torch.int32)), f"{what}: decoded pool differs"
        assert torch.equal(cnt2, cnt)
    return want


def _blob(rng, H, W):
    yy, xx = np.mgrid[:H, :W]
    cy, cx = rng.uniform(0, H), rng.uniform(0, W)
    ry, rx = rng.uniform(0.5, max(H, 2) / 2), rng.uniform(0.5, max(W, 2) / 2)
    m = ((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1
    for _ in range(3):                                               # holes
        y0, x0 = rng.randint(0, H), rng.randint(0, W)
        m[y0:y0 + rng.randint(1, max(H // 4, 2)), x0:x0 + rng.randint(1, max(W // 4, 2))] = False
    return m


def edge_masks(H, W, rng, full=True):
    """Empty, [full], one pixel at each corner, the last column, one row, one column, two far-apart pixels
    (the box is the whole frame), three random blobs."""
    out = []

    def add(*cells, rows=None, cols=None):
        m = np.zeros((H, W), bool)
        for y, x in cells:
            m[y, x] = True
        if rows is not None:
            m[rows, cols] = True
        out.append(m)
    add()
    if full:
        add(rows=slice(None), cols=slice(None))
    for y, x in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1)):
        add((y, x))
    add(rows=slice(None), cols=W - 1)
    add(rows=H // 2, cols=slice(min(1, W - 1), None))
    add(rows=slice(None), cols=W // 3)
    add((0, W - 1), (H - 1, 0))
    for _ in range(3):
        out.append(_blob(rng, H, W))
    return np.stack(out)


def _poison(depth_frames, masks, inst_mask, inst_frame, rays):
    """NaN in every depth pixel outside the masks of the frame's instances and every ray entry outside all
    masks: a read outside an instance's mask, or of another frame, turns its offset into NaN."""
    used = masks[np.asarray(inst_mask)]
    rays[:, ~used.any(0)] = np.nan
    for f in range(len(depth_frames)):
        mine = used[np.asarray(inst_frame) == f]
        depth_frames[f][~mine.any(0)] = np.nan


SHAPES = [(1, 1), (1, 1057), (1057, 1), (37, 100), (29, 1057), (9, 1250), (480, 640), (768, 1024),
          (2048, 2048)]


@pytest.mark.parametrize("H,W", SHAPES, ids=[f"{h}x{w}" for h, w in SHAPES])
def test_offsets_bit_equal_at_frame_edges(H, W):
    """Every edge mask at every frame shape, depth / rays / normals on grids, so every sum is exact: counts and
    offsets bit-equal to the reference.  Instances repeat masks out of order; first one depth frame per
    instance, then five frames dealt at random, each poisoned outside its instances' masks."""
    rng = np.random.RandomState(H * 7919 + W)
    masks = edge_masks(H, W, rng)
    M = len(masks)
    inst_mask = rng.permutation(np.concatenate([np.arange(M), rng.randint(0, M, 3)]))
    n = len(inst_mask)
    normals = _grid(rng, (n, 3), -1, 1, _normal_step(H, W))
    for frames, inst_frame in ((n, rng.permutation(n)), (5, rng.permutation(np.arange(n) % 5))):
        rays = _grid(rng, (3, H, W), -2, 2, 2.0 ** -10)
        depth = _grid(rng, (frames, H, W), 0.5, 4, 2.0 ** -8)
        _poison(depth, masks, inst_mask, inst_frame, rays)
        ref, counts, _, _ = run_case(masks, inst_mask, normals, rays, depth, inst_frame, what=f"{H}x{W} F={frames}")
        assert (counts[inst_mask == 0] == 0).all() and ref[inst_mask == 0].view(np.int32).tolist() == [0] * int(
            (inst_mask == 0).sum())                                   # empty mask: count 0, offset +0.0
        assert (counts[inst_mask == 1] == H * W).all()


def _special_values():
    """(depth, rays (3,), normal (3,)) of the pixels of 1- and 2-pixel instances: non-finite, signed zero,
    denormal and overflowing values, alone and together, then random bit patterns and random fp32 values."""
    big = np.finfo(np.float32).max
    one = [
        (np.nan, (0.5, 0.5, 0.5), (0.25, 0.5, 0.75)),
        (np.inf, (0.5, 0.25, 1.0), (0.25, 0.5, 0.75)),
        (-np.inf, (0.5, 0.25, 1.0), (0.25, 0.5, 0.75)),
        (0.0, (0.5, -0.25, 1.0), (0.25, 0.5, 0.75)),
        (-0.0, (0.5, -0.25, 1.0), (0.25, 0.5, 0.75)),
        (1.0, (-0.0, -0.0, -0.0), (1.0, 1.0, 1.0)),
        (1e-45, (1.0, 0.0, 0.0), (1.0, 0.0, 0.0)),                     # denormal product, term and mean
        (-1e-40, (1.0, 0.0, 0.0), (1.0, 0.0, 0.0)),
        (1.0, (1e-45, 0.0, 0.0), (1.0, 0.0, 0.0)),                     # denormal ray
        (1.0, (1.0, 0.0, 0.0), (-1e-40, 0.0, 0.0)),                    # denormal normal
        (0.5, (1e-38, 0.0, 0.0), (0.75, 0.0, 0.0)),                    # products that round into denormals
        (big, (1.5, 1.5, 0.5), (1.0, 0.5, 0.0)),                       # X, Y overflow to +inf
        (big, (-1.5, -1.5, 0.5), (1.0, 0.5, 0.0)),                     # ... to -inf
        (big, (1.5, -1.5, 0.5), (0.5, 0.5, 0.5)),                      # +inf + -inf inside one term
        (big, (0.5, 0.25, 1.0), (0.5, 0.5, 0.5)),                      # finite, near the top of the range
    ]
    two = [
        ((np.inf, 1.0), ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)), (0.25, 0.5, 0.75)),
        ((np.inf, -np.inf), ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)), (0.25, 0.5, 0.75)),   # both infinities: NaN
        ((-np.inf, np.nan), ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)), (0.25, 0.5, 0.75)),
        ((1e-45, 1e-45), ((1.0, 0.0, 0.0), (1.0, 0.0, 0.0)), (1.0, 0.0, 0.0)),        # mean 1e-45
        ((1e-45, -1e-45), ((1.0, 0.0, 0.0), (1.0, 0.0, 0.0)), (1.0, 0.0, 0.0)),       # +0
        ((2.0 ** 100, 2.0 ** -100), ((1.0, 0.0, 0.0), (1.0, 0.0, 0.0)), (1.0, 0.0, 0.0)),  # one rounding
        ((big, big), ((0.75, 0.0, 0.0), (0.75, 0.0, 0.0)), (1.0, 0.0, 0.0)),        # fp32 sum would overflow
    ]
    return one, two


def test_offsets_of_special_values():
    """1- and 2-pixel instances, bit-equal for any fp32 inputs: NaN, infinities alone and together, signed zeros,
    denormals (a flush-to-zero build changes them), FLT_MAX depth whose products overflow to +-inf, random bit
    patterns and random fp32 values (an FMA-contracted product changes about one term in six).  Each instance
    has its own pixels and its own depth frame; everything else is NaN."""
    rng = np.random.RandomState(11)
    one, two = _special_values()
    normals = [nrm for _, _, nrm in one] + [nrm for _, _, nrm in two]
    cases = [[(d, r)] for d, r, _ in one] + [list(zip(d, r)) for d, r, _ in two]
    bits = rng.randint(0, 1 << 32, size=(384, 2, 7), dtype=np.uint64).astype(np.uint32).view(np.float32)
    conts = np.concatenate([rng.uniform(0.5, 4, (256, 2, 1)), rng.uniform(-2, 2, (256, 2, 3)),
                            rng.uniform(-1, 1, (256, 2, 3))], axis=2).astype(np.float32)
    for k, v in enumerate(np.concatenate([bits, conts])):
        npx = 1 + k % 2
        cases.append([(v[j, 0], tuple(v[j, 1:4])) for j in range(npx)])
        normals.append(tuple(v[0, 4:7]))
    H, W = 8, 1057
    n = len(cases)
    corners = [W - 1, H * W - 1, 0, (H - 1) * W]                      # in the last, partial word column too
    cells = np.concatenate([corners, rng.choice(np.setdiff1d(np.arange(H * W), corners),
                                                size=sum(len(c) for c in cases) - 4, replace=False)])
    masks = np.zeros((n, H, W), bool)
    rays = np.full((3, H * W), np.nan, np.float32)
    depth = np.full((n, H * W), np.nan, np.float32)
    k = 0
    for i, c in enumerate(cases):
        for d, r in c:
            masks[i].reshape(-1)[cells[k]] = True
            depth[i, cells[k]] = d
            rays[:, cells[k]] = r
            k += 1
    ref, counts, bitwise, _ = run_case(masks, np.arange(n), np.array(normals, np.float32), rays.reshape(3, H, W),
                                       depth.reshape(n, H, W), np.arange(n), what="special values")
    assert bitwise.all() and set(counts.tolist()) == {1, 2}
    m = len(one)
    assert np.isnan(ref[[0, 13, m + 1, m + 2]]).all()
    assert ref[[1, 11, m]].tolist() == [np.inf] * 3 and ref[[2, 12]].tolist() == [-np.inf] * 2
    assert ref[[3, 4, 5, m + 4]].view(np.int32).tolist() == [0] * 4          # +0, never -0
    tiny = ref[[6, 7, 8, 9, 10, m + 3]]
    assert ((tiny != 0) & (np.abs(tiny) < np.finfo(np.float32).tiny)).all()   # denormal results
    assert np.isfinite(ref[[14, m + 6]]).all()
    assert np.isnan(ref[len(one) + len(two):]).sum() > 5                    # random bits hit NaN / inf too


def test_offsets_of_cancelling_terms():
    """Mixed-sign terms cancelling to a mean near 0: row 1 mirrors row 0's rays, so the terms cancel in pairs
    but for one pixel whose depth differs by 2^-8.  On grids the sum is exact (bit-equal); with random fp32
    values the result is all rounding error, and must stay within the fp64 summation bound."""
    H, W = 2, 1057
    masks = np.ones((1, H, W), bool)
    rng = np.random.RandomState(5)
    for grid in (True, False):
        if grid:
            r0, d0 = _grid(rng, (3, W), -2, 2, 2.0 ** -10), _grid(rng, (W,), 0.5, 4, 2.0 ** -8)
            nrm = _grid(rng, (2, 3), -1, 1, 2.0 ** -12)
        else:
            r0 = rng.uniform(-2, 2, (3, W)).astype(np.float32)
            d0 = rng.uniform(0.5, 4, W).astype(np.float32)
            nrm = rng.uniform(-1, 1, (2, 3)).astype(np.float32)
        rays = np.stack([r0, -r0], axis=1)
        depth = np.stack([d0, d0])[None].repeat(2, 0)
        depth[1, 0, W // 2] += np.float32(2.0 ** -8)
        ref, _, bitwise, abs_sum = run_case(masks, [0, 0], nrm, rays, depth, [0, 1], exact=grid,
                                            what=f"cancelling grid={grid}")
        assert ref[0] == 0 and ref[0].view(np.int32) == 0 and 0 < abs(ref[1]) < 1e-4 and abs_sum[1] > 100


def test_offsets_from_xyz_over_several_frames():
    """The XYZ path (no depth: the rays hold X, Y, Z) over several frames, one call per frame as
    ``override_depth_batch(xyzs=...)`` makes it, each frame's instances a shuffled subset with repeats; the XYZ
    outside the frame's masks is NaN."""
    rng = np.random.RandomState(3)
    H, W = 37, 1057
    masks = edge_masks(H, W, rng, full=False)
    M = len(masks)
    for f in range(4):
        inst_mask = rng.randint(0, M, 9)
        inst_mask[f % 3] = 0                                           # an empty mask in every frame
        xyz = _grid(rng, (3, H, W), -8, 8, 2.0 ** -18)
        xyz[:, ~masks[inst_mask].any(0)] = np.nan
        run_case(masks, inst_mask, _grid(rng, (9, 3), -1, 1, 2.0 ** -12), xyz, what=f"xyz frame {f}")


def test_seventy_thousand_instances():
    """More instances than a grid's y or z dimension holds (65,535): 70,000 instances of 64 tiny masks, masks
    and frames (F = 5) drawn at random."""
    rng = np.random.RandomState(70000)
    H, W = 37, 100
    masks = np.zeros((64, H, W), bool)
    for m in masks[1:]:
        m.reshape(-1)[rng.choice(H * W, size=rng.randint(1, 5), replace=False)] = True
    masks[5] = False
    masks[5, :, W - 1] = True                                           # the last, partial word column
    n = 70000
    inst_mask, inst_frame = rng.randint(0, 64, n), rng.randint(0, 5, n)
    rays = _grid(rng, (3, H, W), -2, 2, 2.0 ** -10)
    depth = _grid(rng, (5, H, W), 0.5, 4, 2.0 ** -8)
    _poison(depth, masks, inst_mask, inst_frame, rays)
    ref, counts, _, _ = run_case(masks, inst_mask, _grid(rng, (n, 3), -1, 1, 2.0 ** -12), rays, depth, inst_frame,
                                 what="70000 instances")
    assert (counts[inst_mask == 5] == H).all() and (ref[inst_mask == 0].view(np.int32) == 0).all()


def test_abi_refusals_write_nothing():
    """``a3d_plane_offsets`` through the C ABI: bad shapes, each required null pointer and depth without
    ``inst_frame`` return A3D_EINVAL and write nothing; ``n_inst == 0`` is a no-op; a real call writes exactly
    ``n_inst`` entries (64 sentinel entries follow)."""
    lib = _lib.load()
    rng = np.random.RandomState(1)
    H, W = 29, 1057
    masks = edge_masks(H, W, rng)
    n = len(masks)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    rays = torch.from_numpy(_grid(rng, (3, H, W), -2, 2, 2.0 ** -10)).to(DEV)
    depth = torch.from_numpy(_grid(rng, (2, H, W), 0.5, 4, 2.0 ** -8)).to(DEV)
    normals = torch.from_numpy(_grid(rng, (n, 3), -1, 1, 2.0 ** -12)).to(DEV)
    inst_mask = torch.arange(n, dtype=torch.int32, device=DEV)
    inst_frame = torch.from_numpy((np.arange(n) % 2).astype(np.int32)).to(DEV)
    off = torch.full((n + 64,), -7.25, device=DEV)
    cnt = torch.full((n + 64,), -3, dtype=torch.int32, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    args = dict(depth=depth.data_ptr(), rays=rays.data_ptr(), H=H, W=W, bits=pool.bits.data_ptr(),
                bbox=pool.bbox.data_ptr(), inst_mask=inst_mask.data_ptr(), inst_frame=inst_frame.data_ptr(),
                normals=normals.data_ptr(), n_inst=n, offset_out=off.data_ptr(), count_out=cnt.data_ptr())

    def call(**kw):
        a = dict(args, **kw)
        return lib.a3d_plane_offsets(*a.values(), s)

    def untouched(upto=0):
        torch.cuda.synchronize()
        assert off[upto:].eq(-7.25).all() and cnt[upto:].eq(-3).all()

    bad = [dict(n_inst=-1), dict(H=0), dict(H=-5), dict(W=0), dict(W=-1), dict(inst_frame=None)]
    bad += [{k: None} for k in ("rays", "bits", "bbox", "inst_mask", "normals", "offset_out", "count_out")]
    for kw in bad:
        assert call(**kw) == A3D_EINVAL, kw
        assert b"a3d_plane_offsets" in lib.a3d_last_error_string()
    assert call(n_inst=1 << 31) == A3D_ELIMIT
    untouched()
    assert call(n_inst=0) == A3D_OK
    assert call(n_inst=0, depth=None, rays=None, bits=None, bbox=None, inst_mask=None, inst_frame=None,
                normals=None, offset_out=None, count_out=None) == A3D_OK
    untouched()
    assert call() == A3D_OK
    untouched(n)
    assert_offsets(off[:n], cnt[:n], reference(masks, np.arange(n), normals.cpu().numpy(), rays.cpu().numpy(),
                                               depth.cpu().numpy(), np.arange(n) % 2), "abi")
    assert call(depth=None, inst_frame=None, n_inst=n - 1) == A3D_OK                # XYZ path: no frame index
    untouched(n)
    assert_offsets(off[:n - 1], cnt[:n - 1],
                   reference(masks, np.arange(n - 1), normals.cpu().numpy()[:n - 1], rays.cpu().numpy()), "abi xyz")
