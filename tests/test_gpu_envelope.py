"""GPU envelope: the code paths a3d.cu takes only past the shapes of the parity suite, against the C oracle or a
numpy reference — frames wider than 1024 pixels and of 2^20 pixels and more, the limits of the packed arg-max key,
the library's own projection tile, cameras whose K^-1 is not the pinhole pattern, 64-bit mask addressing in
k_score, frames that do not fit shared memory, and the pack kernels at their edge values and grid-stride wraps.

Bit-exact like the parity suite: projected masks word for word, the whole intersection table, unions, arg-max
indices and the IoU bits.  The largest-tile and shared-memory expectations are those of a B200 (227 KiB of
opt-in shared memory per block)."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, geometry, rle
from oracle import c_oracle

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
A3D_ELIMIT = -3
B200_SMEM_OPTIN = 227 * 1024


@pytest.fixture(autouse=True, params=["exact", "filter"])
def projection_kernel(request, monkeypatch):
    """Every test runs with both projection kernels: the reference chain for every point, and the homography
    filter with proven truncation."""
    monkeypatch.setenv("A3D_PROJECT_KERNEL", request.param)
    # fresh pass buffers hold 0xAB bytes: nothing may depend on what a workspace buffer held before
    monkeypatch.setenv("A3D_WS_POISON", "1")
    return request.param


def _unpack(bits: torch.Tensor, W: int) -> np.ndarray:
    """(n,H,pitch) int32 device -> (n,H,W) bool numpy"""
    b = bits.cpu().numpy().view(np.uint32)
    u8 = b.view(np.uint8).reshape(b.shape[0], b.shape[1], -1)
    return np.unpackbits(u8, axis=-1, bitorder="little")[..., :W].astype(bool)


def _bbox_ref(m: np.ndarray):
    if not m.any():
        return [0, -1, 0, -1]
    rows = np.where(m.any(1))[0]
    cols = np.where(m.any(0))[0]
    return [rows[0], rows[-1], cols[0] // 32, cols[-1] // 32]


def _bbox_words(w: np.ndarray):
    """Box of one packed (H, pitch) mask in rows and words."""
    if not w.any():
        return [0, -1, 0, -1]
    rows = np.where(w.any(1))[0]
    cols = np.where(w.any(0))[0]
    return [rows[0], rows[-1], cols[0], cols[-1]]


def _rotations(rng, A, max_angle):
    ax = rng.randn(A, 3)
    ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    ang = rng.uniform(-max_angle, max_angle, A)
    return geometry._axis_angle_to_matrix(torch.from_numpy(ax * ang[:, None])).to(torch.float32).numpy().reshape(A, 9)


def _set_score_kernel(monkeypatch, kernel):
    """kernel: None (the library's choice), ldg | tma | mma, or ldg-addr64 (k_score with 64-bit mask addresses)."""
    if kernel is None:
        monkeypatch.delenv("A3D_SCORE_KERNEL", raising=False)
        return
    monkeypatch.setenv("A3D_SCORE_KERNEL", kernel.split("-")[0])
    if kernel.endswith("-addr64"):
        monkeypatch.setenv("A3D_SCORE_ADDR", "wide")


def _assert_same_iou(got, want):
    """fp32 IoUs bit for bit; a 0/0 is NaN on both sides (its sign and payload differ between the device and
    the host's divide)."""
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _check_against_oracle(res, batch, bits, want_proj, H, W):
    """Every job of a pass against the C oracle: projected masks, counts and boxes, the intersection table,
    unions, arg-max and the IoU bits.  want_proj[j]: the oracle's (A, H, pitch) masks of job j."""
    got_all = res.masks().cpu().numpy().view(np.uint32)
    popc_all, bbox_all = res.proj_popc.cpu().numpy(), res.proj_bbox.cpu().numpy()
    tab_all = res.inter_tab.cpu().numpy()
    cand_all, inter_all, union_all = (t.cpu().numpy() for t in (res.best_cand, res.best_inter, res.best_union))
    iou_all = res.best_iou.cpu().numpy()
    for j, jb in enumerate(batch.jobs):
        A, T = int(jb["n_cand"]), int(jb["n_tgt"])
        c0, t0, b0 = int(jb["cand_begin"]), int(jb["tgt_begin"]), int(jb["tab_begin"])
        proj = want_proj[j]
        diff = int(np.count_nonzero(got_all[c0:c0 + A] != proj))
        assert diff == 0, f"job {j}: {diff} projected words differ"
        assert np.array_equal(popc_all[c0:c0 + A], np.unpackbits(proj.view(np.uint8), axis=None).reshape(A, -1).sum(1))
        assert bbox_all[c0:c0 + A].tolist() == [_bbox_words(p) for p in proj], j
        tg = batch.tgt_index[t0:t0 + T]
        inter, uni, best, iou = c_oracle.score(H, W, bits[tg], proj)
        assert np.array_equal(tab_all[b0:b0 + T * A].reshape(T, A), inter), j
        assert np.array_equal(cand_all[t0:t0 + T], best), j
        assert np.array_equal(inter_all[t0:t0 + T], inter[np.arange(T), best]), j
        assert np.array_equal(union_all[t0:t0 + T], uni[np.arange(T), best]), j
        _assert_same_iou(iou_all[t0:t0 + T], iou)


# ---------------------------------------------------------------------------------------------------------------
# 1. frames past 1024-pixel rows and around 2^20 pixels, through run_pass
# ---------------------------------------------------------------------------------------------------------------
# (W, H) -> (pitch in words, largest projection tile with one-CTA scheduling, packed arg-max key)
LARGE_SHAPES = {
    (1280, 720): (40, 2, True),
    (1025, 1023): (36, 1, True),       # 2^20 - 1 pixels: the last frame of the packed key
    (1024, 1024): (32, 1, False),      # 2^20 pixels: the first frame of the wide key
    (1280, 1024): (40, 1, False),
    (1440, 1080): (48, 1, False),      # the largest common 4:3 frame whose mask fits shared memory
}
IDENTITY_CAND = 2                      # job 0's candidate that maps every pixel onto itself

_large_cache: dict = {}


def _large_case(W, H):
    """Masks, jobs and the oracle's projections of one large frame (built once per shape).

    Job 0 translates the full-frame mask on a fronto-parallel plane; its candidate IDENTITY_CAND shifts by half
    a pixel, so every pixel lands on itself and the full-frame target meets a full-frame candidate: an
    intersection of W*H pixels, 2^20 - 1 at 1025x1023 (the whole 20-bit count field of the packed key) and
    2^20 at 1024x1024 (one more than it holds)."""
    key = (W, H)
    if key in _large_cache:
        return _large_cache[key]
    rng = np.random.RandomState(W * 7 + H)
    cfg = OptConfig.scaled(W, H)
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.zeros((6, H, W), np.float32)
    masks[0] = 1                                                     # full frame
    masks[1, 3:H - 3, 3:W - 3] = 1                                   # near full, with a hole
    masks[1][((yy - H / 3) / 40) ** 2 + ((xx - W / 3) / 60) ** 2 < 1] = 0
    masks[2] = ((yy - H / 2) / (0.3 * H)) ** 2 + ((xx - W / 2) / (0.25 * W)) ** 2 < 1
    masks[3] = ((yy - 0.7 * H) / (0.3 * H)) ** 2 + ((xx - W) / (0.2 * W)) ** 2 < 1   # touches the last column
    box = (np.abs(yy - 0.4 * H) < 0.2 * H) & (np.abs(xx - 0.6 * W) < 0.3 * W)
    masks[4] = box & (rng.rand(H, W) < 0.5)                          # salt and pepper
    # masks[5] stays empty
    bits = c_oracle.pack(masks)
    f = float(cfg.focal_length)
    specs = []
    # job 0: TRANSLATE, full-frame source on the plane z = 2
    off = 2.0
    xf = np.zeros((6, 12), np.float32)
    xf[:, [0, 4, 8]] = 1
    xf[:, 9:] = (rng.randn(6, 3) * 0.05).astype(np.float32)
    xf[IDENTITY_CAND, 9:] = [0.5 * off / f, 0.5 * off / f, 0.0]
    specs.append((0, _lib.MODE_TRANSLATE, np.array([0, 0, 1], np.float32), off, np.zeros(3, np.float32), xf,
                  [0, 1, 2, 3, 5]))
    # job 1: SEQ, near-full source, small rotations about a pivot on the plane
    n1 = np.array([0.1, -0.15, 1.0]) / np.linalg.norm([0.1, -0.15, 1.0])
    xf = np.zeros((8, 12), np.float32)
    xf[:, :9] = _rotations(rng, 8, 0.05)
    specs.append((1, _lib.MODE_SEQ, n1.astype(np.float32), 2.5, np.array([0.1, 0.0, 2.5], np.float32), xf,
                  [1, 0, 4, 2]))
    # job 2: COMPOSED, the blob on the right edge
    xf = np.zeros((8, 12), np.float32)
    xf[:, :9] = _rotations(rng, 8, 0.3)
    xf[:, 9:] = (rng.randn(8, 3) * 0.1).astype(np.float32)
    n2 = np.array([-0.2, 0.1, 1.0]) / np.linalg.norm([-0.2, 0.1, 1.0])
    specs.append((3, _lib.MODE_COMPOSED, n2.astype(np.float32), 3.0, np.zeros(3, np.float32), xf, [3, 2, 5, 0]))
    # job 3: SEQ, the salt-and-pepper source
    xf = np.zeros((5, 12), np.float32)
    xf[:, :9] = _rotations(rng, 5, 0.2)
    specs.append((4, _lib.MODE_SEQ, n1.astype(np.float32), 2.0, np.array([0.0, 0.2, 2.0], np.float32), xf, [4, 1]))
    want = [c_oracle.project(cfg.K_inv(), cfg.focal_length, cfg.cx, cfg.cy, H, W, bits[s[0]], s[2], s[3], s[4],
                             s[1], s[5]) for s in specs]
    full = want[0][IDENTITY_CAND]
    assert np.array_equal(c_oracle.unpack(full[None], W)[0], np.ones((H, W), bool))
    _large_cache[key] = (cfg, masks, bits, specs, want)
    return _large_cache[key]


@pytest.mark.parametrize("plan", ["planned", "uniform"])
@pytest.mark.parametrize("kernel", [None, "ldg", "tma", "mma", "ldg-addr64"])
@pytest.mark.parametrize("W,H", list(LARGE_SHAPES))
def test_large_frames_match_oracle(W, H, kernel, plan, monkeypatch):
    pitch, tile, packed = LARGE_SHAPES[(W, H)]
    assert _lib.pitch_words(W) == pitch
    assert torch.cuda.get_device_properties(0).shared_memory_per_block_optin == B200_SMEM_OPTIN
    monkeypatch.delenv("A3D_PROJECT_SCHED", raising=False)
    assert _lib.load().a3d_project_max_tile(H, W) == tile
    assert (H * W < (1 << 20)) == packed
    _set_score_kernel(monkeypatch, kernel)
    if plan == "uniform":
        monkeypatch.setenv("A3D_TILE_PLAN", "uniform")
    cfg, masks, bits, specs, want = _large_case(W, H)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    assert np.array_equal(pool.bits.cpu().numpy().view(np.uint32), bits)
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    res = engine.run_pass(cfg, pool, engine.DeviceBatch(batch, DEV), want_table=True)
    torch.cuda.synchronize()
    _check_against_oracle(res, batch, bits, want, H, W)
    # the full-frame target's winner is the full-frame candidate, with all W*H pixels in common
    assert res.best_cand[0].item() == IDENTITY_CAND
    assert res.best_inter[0].item() == H * W and res.best_iou[0].item() == 1.0


@pytest.mark.parametrize("sched", ["cta", "persistent"])
@pytest.mark.parametrize("npts", [4095, 8191, 8185, 16383, 8192])
def test_source_whose_last_point_item_is_partial(npts, sched, monkeypatch):
    """The projection takes a source's points 8 at a time, in rounds of one item per thread (1024 threads per CTA,
    512 per persistent group).  When the item count is a multiple of the round but the last item holds fewer
    than 8 points (8191 = 1024 * 8 - 1), that item must still be treated as partial: its unwritten slot is not
    a point."""
    monkeypatch.setenv("A3D_PROJECT_SCHED", sched)
    H, W = 480, 640
    cfg = OptConfig()
    m = np.zeros((2, H * W), np.float32)
    m[0, np.random.RandomState(npts).choice(H * W // 2, npts, replace=False) + H * W // 4] = 1
    m[1, H * W // 3: H * W // 3 + 50000] = 1
    masks = m.reshape(2, H, W)
    bits = c_oracle.pack(masks)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    assert pool.source_points[0] == npts
    rng = np.random.RandomState(1)
    specs = []
    for mode in (_lib.MODE_SEQ, _lib.MODE_COMPOSED, _lib.MODE_TRANSLATE):
        xf = np.zeros((3, 12), np.float32)
        xf[:, :9] = _rotations(rng, 3, 0.2)
        xf[:, 9:] = (rng.randn(3, 3) * 0.05).astype(np.float32)
        specs.append((0, mode, np.array([0, 0, 1], np.float32), 2.0, np.array([0, 0, 2], np.float32), xf, [0, 1]))
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    res = engine.run_pass(cfg, pool, engine.DeviceBatch(batch, DEV), want_table=True, tile_cand=1)
    torch.cuda.synchronize()
    want = [c_oracle.project(cfg.K_inv(), cfg.focal_length, cfg.cx, cfg.cy, H, W, bits[s[0]], s[2], s[3], s[4], s[1],
                             s[5]) for s in specs]
    _check_against_oracle(res, batch, bits, want, H, W)


# ---------------------------------------------------------------------------------------------------------------
# 2. arg-max key limits: a3d_score on candidate masks built by hand
# ---------------------------------------------------------------------------------------------------------------
def _score_only(H, W, tgt_dense, cand_dense, jobs_spec):
    """a3d_score over hand-built masks.  jobs_spec: [(cand_begin, n_cand, [target indices])].
    Returns the result rows and the device inter_tab as numpy."""
    lib = _lib.load()
    tp = engine.pack_masks(torch.from_numpy(tgt_dense).to(DEV))
    cp = engine.pack_masks(torch.from_numpy(cand_dense).to(DEV))
    jobs = np.zeros(len(jobs_spec), _lib.JOB_DTYPE)
    t = tab = 0
    for j, (c0, nc, tg) in enumerate(jobs_spec):
        jobs[j]["cand_begin"], jobs[j]["n_cand"] = c0, nc
        jobs[j]["tgt_begin"], jobs[j]["n_tgt"] = t, len(tg)
        jobs[j]["tab_begin"] = tab
        t += len(tg)
        tab += nc * len(tg)
    tgt_index = np.concatenate([np.asarray(s[2], np.int32) for s in jobs_spec])
    d_jobs = torch.from_numpy(jobs.view(np.uint8).copy()).to(DEV)
    d_tidx = torch.from_numpy(tgt_index).to(DEV)
    nt = len(tgt_index)
    key_ws = torch.full((nt,), -1, dtype=torch.int64, device=DEV)
    inter_tab = torch.full((tab,), -7, dtype=torch.int32, device=DEV)
    out = torch.full((4, nt), -7, dtype=torch.int32, device=DEV)
    _lib.check(lib.a3d_score(H, W, d_jobs.data_ptr(), len(jobs), int(jobs["n_tgt"].max()), int(jobs["n_cand"].max()),
                             nt, len(tp), len(cp), tp.bits.data_ptr(), tp.popc.data_ptr(), tp.bbox.data_ptr(),
                             d_tidx.data_ptr(), cp.bits.data_ptr(), cp.popc.data_ptr(), cp.bbox.data_ptr(),
                             key_ws.data_ptr(), inter_tab.data_ptr(), out[0].data_ptr(), out[1].data_ptr(),
                             out[2].data_ptr(), out[3].data_ptr(), engine._stream_ptr()), "a3d_score")
    torch.cuda.synchronize()
    return jobs, tgt_index, out.cpu().numpy(), inter_tab.cpu().numpy()


def _check_scores(jobs, tgt_index, out, tab, tgt_dense, cand_dense):
    """numpy int64 inter / union, torch's fp32 divide and argmax (first maximum, NaN on top)."""
    tflat = tgt_dense.reshape(len(tgt_dense), -1)
    cflat = cand_dense.reshape(len(cand_dense), -1)
    winners = []
    for jb in jobs:
        c0, A, t0, T, b0 = (int(jb[k]) for k in ("cand_begin", "n_cand", "tgt_begin", "n_tgt", "tab_begin"))
        tm = tflat[tgt_index[t0:t0 + T]]
        cm = cflat[c0:c0 + A]
        inter = tm.astype(np.float32) @ cm.astype(np.float32).T          # exact: counts < 2^24
        inter = inter.astype(np.int64)
        union = tm.sum(1, dtype=np.int64)[:, None] + cm.sum(1, dtype=np.int64)[None, :] - inter
        assert np.array_equal(tab[b0:b0 + T * A].reshape(T, A), inter)
        iou = torch.from_numpy(inter) / torch.from_numpy(union)
        best = iou.argmax(1).numpy()
        sl = slice(t0, t0 + T)
        assert np.array_equal(out[0, sl], best)
        assert np.array_equal(out[1, sl], inter[np.arange(T), best])
        assert np.array_equal(out[2, sl], union[np.arange(T), best])
        _assert_same_iou(out[3, sl].view(np.float32), iou.numpy()[np.arange(T), best])
        winners.append(best)
    return winners


SCORE_KERNELS = ["ldg", "tma", "mma", "ldg-addr64"]


@pytest.mark.parametrize("wc", ["2", "4"])
@pytest.mark.parametrize("kernel", SCORE_KERNELS)
@pytest.mark.parametrize("n_cand", [4096, 4097])
def test_key_candidate_limit(n_cand, kernel, wc, monkeypatch):
    """4096 candidates with the unique winner at 4095 (packed key, its 12-bit candidate field at 0) and 4097 with
    the winner at 4096 (the library must switch to the wide key by itself), on a 100x64 frame."""
    _set_score_kernel(monkeypatch, kernel)
    monkeypatch.setenv("A3D_SCORE_WC", wc)
    monkeypatch.delenv("A3D_SCORE_KEY", raising=False)
    H, W = 64, 100
    rng = np.random.RandomState(n_cand)
    yy, xx = np.mgrid[0:H, 0:W]
    tgt = np.zeros((2, H, W), bool)
    tgt[0] = ((yy - 30) / 20) ** 2 + ((xx - 45) / 35) ** 2 < 1
    tgt[1] = rng.rand(H, W) < 0.3
    inside, outside = np.flatnonzero(tgt[0]), np.flatnonzero(~tgt[0])
    cand = np.repeat(tgt[0].reshape(1, -1), n_cand, axis=0)
    for i in range(n_cand - 1):                       # every other candidate: pixels lost and gained, IoU < 1
        cand[i, rng.choice(inside, 1 + i % 97, replace=False)] = False
        cand[i, rng.choice(outside, i % 13, replace=False)] = True
    cand = cand.reshape(n_cand, H, W)
    jobs, tidx, out, tab = _score_only(H, W, tgt, cand, [(0, n_cand, [0, 1, 0])])
    best = _check_scores(jobs, tidx, out, tab, tgt, cand)[0]
    assert best[0] == n_cand - 1 and best[2] == n_cand - 1


def _fp32_iou_pairs(P, lo_frac=0.9):
    """IoUs k / (P + e) of candidates that hold k of a P-pixel target's pixels and e pixels outside it:
    (k1, 0) and (k2, e2) with different ratios but equal fp32 quotients, and (k3, e3) one fp32 ulp above."""
    f32 = np.float32
    for k1 in range(int(lo_frac * P), int(lo_frac * P) + 4000):
        v = f32(k1) / f32(P)
        e = np.arange(1, 3000)
        k = np.rint(k1 * (P + e) / P).astype(np.int64)
        q = k.astype(f32) / (P + e).astype(f32)
        hit = np.flatnonzero((q == v) & (k * P != k1 * (P + e)) & (k <= P))
        if not len(hit):
            continue
        e2, k2 = int(e[hit[0]]), int(k[hit[0]])
        up = np.nextafter(v, f32(2))
        k_up = np.ceil(up * (P + e)).astype(np.int64)
        qu = k_up.astype(f32) / (P + e).astype(f32)
        hit = np.flatnonzero((qu == up) & (k_up <= P))
        if not len(hit):
            continue
        return (k1, 0), (k2, e2), (int(k_up[hit[0]]), int(e[hit[0]]))
    raise AssertionError("no fp32 IoU tie found")


@pytest.mark.parametrize("wc", ["2", "4"])
@pytest.mark.parametrize("kernel", SCORE_KERNELS)
@pytest.mark.parametrize("W,H", [(1024, 768), (1280, 1024)])
def test_key_ties_nan_and_zero(W, H, kernel, wc, monkeypatch):
    """On both sides of 2^20 pixels (packed and wide key): exact ties and different (inter, union) with equal fp32
    IoUs go to the first candidate, one ulp more to the later one; all-zero IoUs give candidate 0; a 0/0 NaN in the
    middle of the list wins as it does in torch.argmax."""
    _set_score_kernel(monkeypatch, kernel)
    monkeypatch.setenv("A3D_SCORE_WC", wc)
    monkeypatch.delenv("A3D_SCORE_KEY", raising=False)
    P = 500_000
    (k1, e1), (k2, e2), (k3, e3) = _fp32_iou_pairs(P)
    f32 = np.float32
    assert f32(k1) / f32(P + e1) == f32(k2) / f32(P + e2) and k1 * (P + e2) != k2 * (P + e1)
    assert f32(k3) / f32(P + e3) == np.nextafter(f32(k1) / f32(P + e1), f32(2))
    N = H * W

    def mask(k, e):                                   # k of the target's pixels (raster order), e past it
        m = np.zeros(N, bool)
        m[:k] = True
        m[P:P + e] = True
        return m

    tgt = np.zeros((2, N), bool)
    tgt[0, :P] = True                                 # target 1 stays empty
    A, B, U = mask(k1, e1), mask(k2, e2), mask(k3, e3)
    low, low2 = mask(k1 - 5000, 0), mask(k1 - 200, 40)
    empty, outside = np.zeros(N, bool), mask(0, 7000)
    cands = [low, A, B, low2,               # job 0: equal fp32 IoU, A first -> 1
             B, A,                          # job 1: equal fp32 IoU, B first -> 0
             low, A, A.copy(), low2, A,     # job 2: exact ties -> 1
             A, low, U,                     # job 3: one ulp higher and later -> 2
             outside, empty, outside,       # job 4: all IoU zero -> 0
             outside, low, empty, A, empty]  # job 5 on the empty target: 0/0 at 2 -> 2
    starts = np.cumsum([0, 4, 2, 5, 3, 3])
    spec = [(int(starts[0]), 4, [0]), (int(starts[1]), 2, [0]), (int(starts[2]), 5, [0]), (int(starts[3]), 3, [0]),
            (int(starts[4]), 3, [0]), (int(starts[5]), 5, [1, 0])]
    cand = np.stack(cands).reshape(-1, H, W)
    tgt = tgt.reshape(2, H, W)
    jobs, tidx, out, tab = _score_only(H, W, tgt, cand, spec)
    win = _check_scores(jobs, tidx, out, tab, tgt, cand)
    assert [int(w[0]) for w in win] == [1, 0, 1, 2, 0, 2]
    assert np.isnan(out[3, 5:6].view(np.float32)[0])             # job 5, empty target


# ---------------------------------------------------------------------------------------------------------------
# 3. general intrinsics: K^-1 other than [[a,0,b],[0,c,d],[0,0,1]]
# ---------------------------------------------------------------------------------------------------------------
def _rot(axis, deg):
    a = np.asarray(axis, np.float64)
    return geometry._axis_angle_to_matrix(torch.from_numpy(a / np.linalg.norm(a) * math.radians(deg))).numpy().reshape(3, 3)


def _general_kinv(kind, cfg):
    K0 = cfg.K()
    if kind == "skewed":                    # non-square pixels, skew, principal point off centre
        K = np.array([[cfg.focal_length * 1.05, 12.0, cfg.cx + 7.0],
                      [0.0, cfg.focal_length * 0.93, cfg.cy - 5.0],
                      [0.0, 0.0, 1.0]])
        return np.linalg.inv(K)
    if kind == "rotated":                   # camera rotated by 4 degrees: kinv[6], kinv[7] != 0, kinv[8] != 1
        return _rot([0.3, 1.0, 0.2], 4.0) @ np.linalg.inv(K0)
    # grazing: tilted about x so that the rays of the rows near 10 % of the height lie in the plane z = const
    ry = (0.1 * cfg.height - cfg.cy) / cfg.focal_length
    return _rot([1.0, 0.1, 0.0], math.degrees(math.atan(-1.0 / ry))) @ np.linalg.inv(K0)


@pytest.mark.parametrize("W,H", [(640, 480), (1280, 720)])
@pytest.mark.parametrize("kind", ["skewed", "rotated", "grazing"])
def test_general_intrinsics_match_oracle(kind, W, H, monkeypatch):
    cfg = OptConfig.scaled(W, H)
    kinv = _general_kinv(kind, cfg)
    assert not (kinv[0, 1] == 0 and kinv[1, 0] == 0 and kinv[2, 0] == 0 and kinv[2, 1] == 0 and kinv[2, 2] == 1)
    if kind != "skewed":
        assert kinv[2, 0] != 0 and kinv[2, 1] != 0 and kinv[2, 2] != 1
    rz = kinv[2, 0] * np.arange(W)[None, :] + kinv[2, 1] * np.arange(H)[:, None] + kinv[2, 2]
    assert (rz.min() < 0 < rz.max()) == (kind == "grazing")          # the plane z = const contains some rays
    cam = _lib.Camera()
    for i, v in enumerate(kinv.reshape(-1)):
        cam.kinv[i] = float(v)
    cam.f, cam.cx, cam.cy, cam.H, cam.W = float(cfg.focal_length), float(cfg.cx), float(cfg.cy), H, W
    monkeypatch.setattr(engine, "_camera_cached", lambda c: cam)
    rng = np.random.RandomState(len(kind) * 1000 + W)
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.zeros((5, H, W), np.float32)
    masks[0, 2:H - 2, 2:W - 2] = 1
    for i in range(1, 4):
        cy, cx = rng.uniform(0.2, 0.8) * H, rng.uniform(0.2, 0.8) * W
        masks[i] = ((yy - cy) / (rng.uniform(0.1, 0.4) * H)) ** 2 + ((xx - cx) / (rng.uniform(0.1, 0.4) * W)) ** 2 < 1
    masks[3] *= rng.rand(H, W) < 0.6
    masks[4, :H // 5] = 1                                            # the rows around the grazing rays
    bits = c_oracle.pack(masks)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    specs = []
    for j, (mode, src) in enumerate([(_lib.MODE_SEQ, 0), (_lib.MODE_COMPOSED, 1), (_lib.MODE_TRANSLATE, 2),
                                     (_lib.MODE_SEQ, 4), (_lib.MODE_COMPOSED, 3), (_lib.MODE_TRANSLATE, 4)]):
        A = 16
        xf = np.zeros((A, 12), np.float32)
        xf[:, :9] = _rotations(rng, A, 0.5) if mode != _lib.MODE_TRANSLATE else np.eye(3, dtype=np.float32).reshape(9)
        xf[:, 9:] = (rng.randn(A, 3) * 0.2).astype(np.float32)
        normal = np.array([0.0, 0.0, 1.0]) if j >= 3 else np.array([0.1, -0.2, 1.0]) + 0.05 * rng.randn(3)
        normal = (normal / np.linalg.norm(normal)).astype(np.float32)
        pivot = (rng.randn(3) * 0.3 + [0, 0, 2]).astype(np.float32)
        specs.append((src, mode, normal, 2.0, pivot, xf, [0, 1, 2, 3, 4]))
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    res = engine.run_pass(cfg, pool, engine.DeviceBatch(batch, DEV), want_table=True)
    torch.cuda.synchronize()
    want = [c_oracle.project(kinv, cfg.focal_length, cfg.cx, cfg.cy, H, W, bits[s[0]], s[2], s[3], s[4], s[1], s[5])
            for s in specs]
    assert sum(int(w.any()) for w in want) == len(specs)
    _check_against_oracle(res, batch, bits, want, H, W)


# ---------------------------------------------------------------------------------------------------------------
# 5. limits are refused cleanly
# ---------------------------------------------------------------------------------------------------------------
def _small_pass():
    """An ordinary 640x480 pass (the same each call) and its results."""
    cfg = OptConfig()
    H, W = cfg.height, cfg.width
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.stack([((yy - 200) / 90.0) ** 2 + ((xx - 300) / 120.0) ** 2 < 1,
                      ((yy - 260) / 80.0) ** 2 + ((xx - 340) / 110.0) ** 2 < 1]).astype(np.float32)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    xf = np.zeros((6, 12), np.float32)
    xf[:, :9] = _rotations(np.random.RandomState(3), 6, 0.3)
    batch = engine.build_batch([0], [_lib.MODE_SEQ], [np.array([0, 0, 1], np.float32)], [2.0],
                               [np.array([0, 0, 2], np.float32)], [xf], [[0, 1]], pool.source_points)
    res = engine.run_pass(cfg, pool, engine.DeviceBatch(batch, DEV), want_table=True)
    torch.cuda.synchronize()
    return [t.cpu().numpy().copy() for t in (res.masks(), res.inter_tab, res.best_cand, res.best_inter)]


def _assert_still_works(before):
    after = _small_pass()
    torch.cuda.synchronize()
    for a, b in zip(before, after):
        assert np.array_equal(a, b)


def test_frames_over_shared_memory_are_refused():
    """1920x1080: a3d_project_max_tile, a3d_project and a3d_pass return A3D_ELIMIT naming the shape, run_pass
    raises; a3d_rle_to_bits refuses frames over its own limit.  The stream stays usable after each refusal."""
    lib = _lib.load()
    before = _small_pass()
    H, W = 1080, 1920
    shape = f"{H}x{W}"
    assert lib.a3d_project_max_tile(H, W) == A3D_ELIMIT
    assert shape in lib.a3d_last_error_string().decode()
    _assert_still_works(before)
    cfg = OptConfig.scaled(W, H)
    cam = engine.camera_struct(cfg)
    buf = torch.zeros(1 << 16, dtype=torch.int64, device=DEV)
    p = buf.data_ptr()
    s = engine._stream_ptr()
    rc = lib.a3d_project(C.byref(cam), p, 1, 1, 0, p, p, p, p, p, p, None, 0, p, p, p, _lib.OUT_FULL, s)
    assert rc == A3D_ELIMIT and shape in lib.a3d_last_error_string().decode()
    _assert_still_works(before)
    rc = lib.a3d_pass(C.byref(cam), p, 1, 1, 1, 0, 1, 1, 1, p, p, p, p, p, p, p, p, p, p, None, 0, p, p, p, p, p,
                      p, p, p, p, _lib.OUT_FULL, s)
    assert rc == A3D_ELIMIT and shape in lib.a3d_last_error_string().decode()
    _assert_still_works(before)
    m = np.zeros((1, H, W), np.float32)
    m[0, 100:300, 200:900] = 1
    pool = engine.pack_masks(torch.from_numpy(m).to(DEV))
    xf = np.zeros((2, 12), np.float32)
    xf[:, [0, 4, 8]] = 1
    batch = engine.build_batch([0], [_lib.MODE_COMPOSED], [np.array([0, 0, 1], np.float32)], [2.0],
                               [np.zeros(3, np.float32)], [xf], [[0]], pool.source_points)
    with pytest.raises(_lib.A3DError, match=shape):
        engine.run_pass(cfg, pool, engine.DeviceBatch(batch, DEV), want_table=True)
    _assert_still_works(before)
    # a3d_rle_to_bits keeps 8 KiB of shared memory for itself: 1440x1200 fits the projection, not the decoder
    assert lib.a3d_project_max_tile(1200, 1440) == 1
    for h, w in ((1080, 1920), (1200, 1440)):
        assert h * _lib.pitch_words(w) * 4 > B200_SMEM_OPTIN - 8192
        rc = lib.a3d_rle_to_bits(p, p, 1, h, w, p, s)
        assert rc == A3D_ELIMIT and f"{h}x{w}" in lib.a3d_last_error_string().decode()
        _assert_still_works(before)


def test_persistent_schedule_limits_and_default_tile(monkeypatch):
    """Persistent CTAs hold two groups of candidate slots, which halves the largest tile: 1280x1024 no longer
    fits (A3D_ELIMIT), and 1024x768 drops from 2 candidates to 1.  A default-tile run_pass under the persistent
    schedule, after one under the default schedule in the same process, must use the smaller tile and give what
    the default schedule gives, and what the C oracle gives.  4 jobs x 360 candidates: several waves of CTAs,
    where the engine picks uniform tiles of 2 under the default schedule."""
    lib = _lib.load()
    monkeypatch.setenv("A3D_PROJECT_SCHED", "persistent")
    assert lib.a3d_project_max_tile(1024, 1280) == A3D_ELIMIT
    assert "1024x1280" in lib.a3d_last_error_string().decode()
    assert lib.a3d_project_max_tile(768, 1024) == 1
    monkeypatch.setenv("A3D_PROJECT_SCHED", "cta")
    assert lib.a3d_project_max_tile(768, 1024) == 2
    W, H = 1024, 768
    cfg = OptConfig.scaled(W, H)
    rng = np.random.RandomState(11)
    yy, xx = np.mgrid[0:H, 0:W]
    masks = np.stack([((yy - 380) / 150.0) ** 2 + ((xx - 500) / 200.0) ** 2 < 1,
                      ((yy - 300) / 120.0) ** 2 + ((xx - 600) / 180.0) ** 2 < 1,
                      (rng.rand(H, W) < 0.1) & (np.abs(yy - 400) < 200)]).astype(np.float32)
    bits = c_oracle.pack(masks)
    pool = engine.pack_masks(torch.from_numpy(masks).to(DEV))
    specs = []
    for j, mode in enumerate((_lib.MODE_SEQ, _lib.MODE_COMPOSED, _lib.MODE_TRANSLATE, _lib.MODE_SEQ)):
        xf = np.zeros((360, 12), np.float32)
        xf[:, :9] = _rotations(rng, 360, 0.4)
        xf[:, 9:] = (rng.randn(360, 3) * 0.1).astype(np.float32)
        specs.append((j % 3, mode, np.array([0.1, 0.0, 1.0], np.float32) / np.float32(np.hypot(0.1, 1.0)), 2.0,
                      np.array([0, 0, 2], np.float32), xf, [0, 1, 2]))
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    out = {}
    for sched in ("cta", "persistent"):
        monkeypatch.setenv("A3D_PROJECT_SCHED", sched)
        dbatch = engine.DeviceBatch(batch, DEV)
        res = engine.run_pass(cfg, pool, dbatch, want_table=True)
        torch.cuda.synchronize()
        assert dbatch.tile_plan(cfg) == ((2, None) if sched == "cta" else (1, None))
        out[sched] = [t.cpu().numpy().copy() for t in (res.masks(), res.proj_popc, res.proj_bbox, res.inter_tab,
                                                        res.best_cand, res.best_inter, res.best_union)]
        if sched == "persistent":
            want = [c_oracle.project(cfg.K_inv(), cfg.focal_length, cfg.cx, cfg.cy, H, W, bits[s[0]], s[2], s[3],
                                     s[4], s[1], s[5]) for s in specs]
            _check_against_oracle(res, batch, bits, want, H, W)
    for a, b in zip(out["cta"], out["persistent"]):
        assert np.array_equal(a, b)


def test_rle_decode_of_a_large_frame_equals_dense_pack():
    H, W = 1080, 1440
    yy, xx = np.mgrid[0:H, 0:W]
    rng = np.random.RandomState(5)
    ms = [((yy - 500) / 400.0) ** 2 + ((xx - 700) / 650.0) ** 2 < 1,
          (rng.rand(H, W) < 0.1) | (xx == W - 1),
          np.ones((H, W), bool)]
    pool = engine.rle_to_pool([rle.encode(m) for m in ms], H, W, DEV)
    dense = engine.pack_masks(torch.from_numpy(np.stack(ms).astype(np.uint8)).to(DEV))
    assert torch.equal(pool.bits, dense.bits)
    assert torch.equal(pool.popc, dense.popc) and torch.equal(pool.bbox, dense.bbox)
    assert np.array_equal(_unpack(pool.bits, W), np.stack(ms))


# ---------------------------------------------------------------------------------------------------------------
# 6. pack stage against c_oracle.pack and numpy
# ---------------------------------------------------------------------------------------------------------------
def _pack_raw(src: torch.Tensor, n, H, W, thresh, elem_offset=0):
    """a3d_pack_masks on (n, H, W) elements starting elem_offset elements into the flat device tensor src; both
    bit planes into buffers that start out as 0xAB bytes (every word, padding included, must be written)."""
    lib = _lib.load()
    code = {torch.float32: _lib.A3D_F32, torch.uint8: _lib.A3D_U8}[src.dtype]
    pitch = _lib.pitch_words(W)
    gt = torch.full((n, H, pitch), -0x54545455, dtype=torch.int32, device=DEV)
    nz = torch.full_like(gt, -0x54545455)
    _lib.check(lib.a3d_pack_masks(src.data_ptr() + elem_offset * src.element_size(), code, n, H, W, float(thresh),
                                  gt.data_ptr(), nz.data_ptr(), engine._stream_ptr()), "a3d_pack_masks")
    torch.cuda.synchronize()
    return gt.cpu().numpy().view(np.uint32), nz.cpu().numpy().view(np.uint32)


def _edge_values(thresh):
    f32 = np.float32
    t = f32(thresh)
    return np.array([t, np.nextafter(t, f32(1)), np.nextafter(t, f32(-1)), np.nan, -np.nan, np.inf, -np.inf, -0.0,
                     0.0, -1.0, -t, 1.0, 2.0, 1e-45, -1e-45, 0.5, 0.3], np.float32)


@pytest.mark.parametrize("W", [640, 1057])
@pytest.mark.parametrize("thresh", [0.0, 0.3, 0.5])
def test_pack_edge_values_and_alignment(thresh, W):
    """Values at the threshold and one ulp either side, NaN, +-inf, -0.0, negatives and denormals; the vector kernel
    (16-byte aligned rows) and the scalar kernel (the same data 4 bytes off alignment)."""
    n, H = 5, 37
    rng = np.random.RandomState(int(thresh * 10) + W)
    x = rng.choice(_edge_values(thresh), size=(n, H, W)).astype(np.float32)
    x[0, :, -1] = thresh + 1.0                        # last column set / at the threshold
    x[1, :, -1] = thresh
    want_gt = c_oracle.pack(x, thresh)
    want_nz = c_oracle.pack(x, nonzero=True)
    assert np.array_equal(c_oracle.unpack(want_gt.reshape(n * H, 1, -1), W).reshape(n, H, W), x > np.float32(thresh))
    assert np.array_equal(c_oracle.unpack(want_nz.reshape(n * H, 1, -1), W).reshape(n, H, W), x != 0)
    flat = torch.zeros(n * H * W + 4, dtype=torch.float32, device=DEV)
    for off in (0, 1):                                # off 1: 4 bytes past 16-byte alignment -> k_pack
        flat[off:off + n * H * W] = torch.from_numpy(x.reshape(-1)).to(DEV)
        gt, nz = _pack_raw(flat, n, H, W, thresh, off)
        assert np.array_equal(gt, want_gt), off
        assert np.array_equal(nz, want_nz), off
    # through pack_masks: popcounts / boxes of both planes
    pool = engine.pack_masks(torch.from_numpy(x).to(DEV), thresh, with_nonzero=True)
    assert np.array_equal(pool.bits.cpu().numpy().view(np.uint32), want_gt)
    assert pool.bits_nz is not None and np.array_equal(pool.bits_nz.cpu().numpy().view(np.uint32), want_nz)
    assert pool.bbox.cpu().numpy().tolist() == [_bbox_ref(m) for m in x > np.float32(thresh)]
    assert pool.bbox_nz.cpu().numpy().tolist() == [_bbox_ref(m) for m in x != 0]


@pytest.mark.parametrize("W", [1056, 1057])
@pytest.mark.parametrize("thresh", [0.0, 1.5])
def test_pack_uint8(thresh, W):
    n, H = 4, 29
    rng = np.random.RandomState(W)
    x = rng.choice(np.array([0, 1, 2, 255], np.uint8), size=(n, H, W))
    gt, nz = _pack_raw(torch.from_numpy(x.reshape(-1)).to(DEV), n, H, W, thresh)
    assert np.array_equal(gt, c_oracle.pack(x.astype(np.float32), thresh))
    assert np.array_equal(nz, c_oracle.pack(x.astype(np.float32), nonzero=True))
    assert np.array_equal(c_oracle.unpack(gt.reshape(n * H, 1, -1), W).reshape(n, H, W), x > thresh)


@pytest.mark.parametrize("kernel", ["vector", "scalar"])
def test_pack_grid_stride_wraps(kernel):
    """Enough rows that every warp of both pack kernels goes around its grid-stride loop at least twice (the
    grids are capped at 16 CTAs of 8 warps per SM; k_pack_vec takes 4 128-pixel segments per warp step)."""
    warps = torch.cuda.get_device_properties(0).multi_processor_count * 16 * 8
    if kernel == "vector":
        H, W = 480, 640
        n = -(-3 * warps * 4 // (H * ((W + 127) // 128)))
    else:
        H, W = 1000, 1057
        n = -(-3 * warps // H)
    rng = np.random.RandomState(n)
    x = rng.rand(n, H, W).astype(np.float32)
    x[:, :, -1] = 0.75
    gt, nz = _pack_raw(torch.from_numpy(x.reshape(-1)).to(DEV), n, H, W, 0.5)
    assert np.array_equal(gt, c_oracle.pack(x, 0.5))
    assert np.array_equal(nz, c_oracle.pack(x, nonzero=True))


@pytest.mark.parametrize("W", [1057, 1250])
def test_mask_meta_last_column(W):
    """Boxes and counts of masks that touch the last column of frames wider than 1024 with W % 32 != 0."""
    H = 9
    m = np.zeros((5, H, W), bool)
    m[0, 4, W - 1] = True                             # one pixel, last column
    m[1, :, W - 1] = True
    m[2, 2, W - 33:] = True                           # across the last two words
    m[3] = True
    pool = engine.pack_masks(torch.from_numpy(m).to(DEV))
    assert np.array_equal(pool.popc.cpu().numpy(), m.reshape(5, -1).sum(1))
    assert pool.bbox.cpu().numpy().tolist() == [_bbox_ref(x) for x in m]
    assert pool.bbox[0, 3].item() == (W - 1) // 32
