"""Kernels past 2^31 and 2^32 elements of their buffers, where the one-GPU C3 (640x480) and C4 (1024x768) passes run:
a mask pool of 2.4e9 words, projected-mask buffers of 3.5e9 and 9e9 words.  Every kernel that turns a mask, frame,
candidate or table index into an address is run with that index's buffer offset across 2^31 or 2^32 elements, and its
results are compared exactly with the C oracle or the numpy restatements, so that one lost 64-bit cast fails a test.

Layout (640x480, 9,600 words a mask): slot 223,696 straddles word 2^31 (at row 102) and slot 447,392 straddles word
2^32 (at row 204).  A pool of 447,392 masks ends just below 2^32 words, the last size k_score addresses with 32-bit
offsets; one mask more and it takes 64-bit addresses.  One zeroed (447,393, 480, 20) int32 pool (17.2 GB) serves both
sizes; real masks sit near slot 0, around both straddling slots and at the end, and every other slot is empty.
Nothing past a few slots is ever copied to the host: slots are read with index_select, the rest checked on the device.

Each test needs up to about 35 GB of device memory and skips, saying so, when the shared device has less free."""
import ctypes as C
import time
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from articulation3d_b200 import OptConfig, _lib, engine, geometry, rle, synth
from oracle import c_oracle
from tests import plane_maps_ref, render_ref
from tests.test_gpu_plane_offsets import assert_offsets, reference

DEV = "cuda:0"
GiB = 1 << 30
H, W = 480, 640
PITCH = 20
WORDS = H * PITCH                                   # 9,600 32-bit words a mask


# ---------------------------------------------------------------------------------------------------------------
# layout arithmetic (checked on the CPU below)
# ---------------------------------------------------------------------------------------------------------------
def straddling_slot(size: int, boundary: int) -> int:
    """The item of ``size`` elements that holds element ``boundary`` of a buffer of such items."""
    return boundary // size


def boundary_row(slot: int, size: int, row_elems: int, boundary: int) -> int:
    """Row of item ``slot`` that holds element ``boundary``."""
    return (boundary - slot * size) // row_elems


def narrow_limit(words: int) -> int:
    """Largest pool k_score addresses with 32-bit word offsets: n * words < 2^32."""
    return ((1 << 32) - 1) // words


def filler_layout(n_total: int, real, chunk: int = 4096):
    """Jobs that fill [0, n_total) candidate slots: ``real`` is a list of (cand_begin, n_cand), sorted and disjoint;
    the gaps go to filler jobs of at most ``chunk`` candidates.  Returns [(kind, index or None, begin, count)], kind
    'real' or 'filler', in slot order."""
    out, pos = [], 0
    for i, (b, n) in enumerate(real):
        assert b >= pos
        while pos < b:
            k = min(chunk, b - pos)
            out.append(("filler", None, pos, k))
            pos += k
        out.append(("real", i, b, n))
        pos = b + n
    assert pos <= n_total
    while pos < n_total:
        k = min(chunk, n_total - pos)
        out.append(("filler", None, pos, k))
        pos += k
    return out


def table_filler_targets(filler_cand: int, boundary: int) -> int:
    """Targets of a filler of ``filler_cand`` candidates whose table ends less than ``filler_cand`` entries before
    ``boundary``: the next job's table starts just below it."""
    return (boundary - 1) // filler_cand


def pcd_fillers(points: int, planes: int, boundary: int) -> int:
    """Jobs of ``points`` source points to put in front of a job so that its point-cloud slice starts past
    ``boundary`` floats (``planes`` floats a point)."""
    return boundary // (planes * points) + 1


def rle_call_arrays(n: int, hw: int, placed: dict):
    """Flat run lengths and begin[n+1] of n masks for one a3d_rle_to_bits call: ``placed`` maps a mask index to its
    runs, every other mask is empty (one run of hw zeros).  Vectorised: n may be hundreds of thousands."""
    lens = np.ones(n, np.int64)
    for s, c in placed.items():
        lens[s] = len(c)
    begin = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=begin[1:])
    counts = np.full(int(begin[-1]), hw, np.uint32)
    for s, c in placed.items():
        counts[begin[s]:begin[s + 1]] = c
    return counts, begin


S31 = straddling_slot(WORDS, 1 << 31)               # 223,696
S32 = straddling_slot(WORDS, 1 << 32)               # 447,392
N_NARROW = narrow_limit(WORDS)                      # 447,392
N_WIDE = N_NARROW + 1
EMPTY = 5                                           # a slot no mask is written to
FULL = 3                                            # the full-frame mask
PLACED = [0, 1, 2, S31 - 1, S31, S31 + 1] + list(range(S32 - 9, S32 + 1))
FAR = [S32, S31, S32 - 1, S31 + 1, S32 - 9]         # index lists of the per-mask kernels
N_REAL = 180                                        # candidates of a real job
K_STRADDLE = 90                                     # a real job's candidate that sits in a straddling slot
RGB_FRAME = straddling_slot(H * W * 3, 1 << 31)     # 2,330: a frame of RGB bytes across 2^31
F32_FRAME = straddling_slot(H * W, 1 << 31)         # 6,990: a frame of floats across 2^31


def test_boundary_arithmetic():
    assert (S31, S32) == (223_696, 447_392)
    assert S31 * WORDS <= 1 << 31 < (S31 + 1) * WORDS and S32 * WORDS <= 1 << 32 < (S32 + 1) * WORDS
    assert boundary_row(S31, WORDS, PITCH, 1 << 31) == 102 and boundary_row(S32, WORDS, PITCH, 1 << 32) == 204
    assert N_NARROW == 447_392 and N_NARROW * WORDS == 4_294_963_200 < 1 << 32 <= N_WIDE * WORDS
    # C4: 1024x768 masks are 24,576 words; its 368,640 projected slots are past 2^33
    assert narrow_limit(768 * 32) == 174_762 and 368_640 * 768 * 32 > 1 << 33
    assert (RGB_FRAME, F32_FRAME) == (2330, 6990)
    assert boundary_row(RGB_FRAME, H * W * 3, W * 3, 1 << 31) == 81
    assert boundary_row(F32_FRAME, H * W, W, 1 << 31) == 243
    # the contiguous emit of the pool's last 7,000 masks: the placed masks are its outputs 6,990 .. 6,999
    assert N_WIDE - 7000 + F32_FRAME == S32 - 9 and 7000 * H * W > 1 << 31
    t = table_filler_targets(4096, 1 << 31)
    assert t == 524_287 and 4096 * t < 1 << 31 < 4096 * t + 24 * N_REAL
    n = pcd_fillers(H * W, _lib.PCD_PLANES, 1 << 31)
    assert n == 1399 and _lib.PCD_PLANES * n * H * W > 1 << 31 > _lib.PCD_PLANES * (n - 1) * H * W


def test_filler_layout():
    """The pass layouts: the narrow one ends at the last 32-bit-addressable slot, the wide one puts candidate
    K_STRADDLE of its last real job in slot S32."""
    wide_total = S32 - K_STRADDLE + N_REAL
    assert N_NARROW * WORDS < 1 << 32 < wide_total * WORDS
    for n_total, real in ((N_NARROW, [(0, N_REAL), (S31 - K_STRADDLE, N_REAL), (N_NARROW - N_REAL, N_REAL)]),
                          (wide_total, [(0, N_REAL), (S31 - K_STRADDLE, N_REAL), (S32 - K_STRADDLE, N_REAL)])):
        lay = filler_layout(n_total, real)
        assert lay[0][2] == 0 and sum(x[3] for x in lay) == n_total
        assert all(a[2] + a[3] == b[2] for a, b in zip(lay, lay[1:]))
        assert [(x[2], x[3]) for x in lay if x[0] == "real"] == real
        assert all(0 < x[3] <= 4096 for x in lay if x[0] == "filler")
        assert lay[-1][0] == "real" and real[1][0] + K_STRADDLE == S31


def test_rle_call_arrays_match_a_loop():
    hw = 6 * 5
    placed = {3: np.array([0, 4, 26], np.uint32), 7: np.array([2, 28], np.uint32), 49: np.array([30], np.uint32)}
    counts, begin = rle_call_arrays(50, hw, placed)
    flat, b = [], [0]
    for i in range(50):
        flat.extend(placed.get(i, [hw]))
        b.append(len(flat))
    assert begin.dtype == np.int64 and counts.dtype == np.uint32
    assert np.array_equal(begin, b) and np.array_equal(counts, flat)
    assert all(int(counts[begin[i]:begin[i + 1]].sum()) == hw for i in range(50))


# ---------------------------------------------------------------------------------------------------------------
# device fixtures
# ---------------------------------------------------------------------------------------------------------------
def _need(nbytes: int):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + GiB:
        pytest.skip(f"needs {(nbytes + GiB) / GiB:.1f} GiB of free device memory, {free / GiB:.1f} GiB free")


@pytest.fixture
def _measure(request):
    """Wall time and peak device memory of the test, as junit properties."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    torch.cuda.synchronize()
    request.node.user_properties.append(("wall_s", round(time.perf_counter() - t0, 2)))
    request.node.user_properties.append(("peak_alloc_gib", round(torch.cuda.max_memory_allocated() / GiB, 2)))
    torch.cuda.empty_cache()


def gpu(fn):
    return pytest.mark.gpu(pytest.mark.usefixtures("_measure")(fn))


def _placed_masks():
    """slot -> (H, W) bool: masks of a synthetic clip whose rows reach above row 75 and below row 250, so that every
    placed mask has pixels on both sides of the boundary rows (81, 102, 204, 243)."""
    cfg = OptConfig()
    scene = synth.make_scene(7, 2, 12, cfg, kinds=[1, 1])
    ms = np.concatenate([synth.render_track_masks(scene, t, cfg).numpy() for t in range(2)])
    rows = [np.flatnonzero(m.any(1)) for m in ms]
    sel = [m for m, r in zip(ms, rows) if r[0] <= 75 and r[-1] >= 250]
    assert len(sel) >= 8
    out = {s: sel[i % len(sel)] for i, s in enumerate(PLACED)}
    out[FULL] = np.ones((H, W), bool)
    return out


def _straddles(flat_words: np.ndarray, word: int) -> bool:
    return bool(flat_words[:word].any() and flat_words[word:].any())


@pytest.fixture(scope="module")
def big():
    """The (N_WIDE, H, PITCH) pool with the placed masks, its popcounts and boxes, host copies of the placed masks."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    _need(N_WIDE * WORDS * 4)
    masks = _placed_masks()
    slots = sorted(masks)
    packed_host = c_oracle.pack(np.stack([masks[s] for s in slots]).astype(np.float32))
    bits = torch.zeros(N_WIDE, H, PITCH, dtype=torch.int32, device=DEV)
    dense = torch.from_numpy(np.stack([masks[s] for s in slots]).astype(np.uint8)).to(DEV)
    bits.index_copy_(0, torch.tensor(slots, device=DEV), engine.pack_masks(dense).bits)
    del dense
    pool = engine.pool_from_bits(bits, H, W)
    got = bits.index_select(0, torch.tensor(slots, device=DEV)).cpu().numpy().view(np.uint32)
    assert np.array_equal(got, packed_host)
    packed = dict(zip(slots, packed_host))
    assert _straddles(packed[S31].reshape(-1), (1 << 31) - S31 * WORDS)
    assert _straddles(packed[S32].reshape(-1), (1 << 32) - S32 * WORDS)
    ns = SimpleNamespace(cfg=OptConfig(), masks=masks, packed=packed, bits=bits, wide=pool,
                         narrow=engine.MaskPool(bits[:N_NARROW], pool.popc[:N_NARROW], pool.bbox[:N_NARROW], H, W))
    yield ns
    ns.__dict__.clear()
    del bits, pool
    torch.cuda.empty_cache()


def _packed(big, slots) -> np.ndarray:
    return np.stack([big.packed[s] if s in big.packed else np.zeros((H, PITCH), np.uint32) for s in slots])


def _dense(big, slots) -> np.ndarray:
    return np.stack([big.masks[s] if s in big.masks else np.zeros((H, W), bool) for s in slots])


def _all_zero(t: torch.Tensor, step: int = 1 << 14) -> bool:
    """No nonzero element in t (checked on the device, ``step`` rows of t at a time)."""
    return not any(bool(t[a:a + step].any()) for a in range(0, t.shape[0], step))


# ---------------------------------------------------------------------------------------------------------------
# 1. passes against the C oracle on the 447,392-mask (32-bit offsets) and 447,393-mask (64-bit) pools
# ---------------------------------------------------------------------------------------------------------------
def _rotations(rng, A, max_angle):
    ax = rng.randn(A, 3)
    ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    ang = rng.uniform(-max_angle, max_angle, A)
    return geometry._axis_angle_to_matrix(torch.from_numpy(ax * ang[:, None])).to(torch.float32).numpy().reshape(A, 9)


def _xforms(seed, mode, A=N_REAL):
    rng = np.random.RandomState(seed)
    xf = np.zeros((A, 12), np.float32)
    if mode == _lib.MODE_TRANSLATE:
        xf[:, [0, 4, 8]] = 1
        xf[:, 9:] = (rng.randn(A, 3) * 0.05).astype(np.float32)
    else:
        xf[:, :9] = _rotations(rng, A, 0.12)
        xf[:, 9:] = (rng.randn(A, 3) * 0.02).astype(np.float32)
    return xf


def _identity(A):
    xf = np.zeros((A, 12), np.float32)
    xf[:, [0, 4, 8]] = 1
    return xf


Z = np.array([0, 0, 1], np.float32)
N1 = (np.array([0.1, -0.05, 1.0]) / np.linalg.norm([0.1, -0.05, 1.0])).astype(np.float32)


def _real_spec(which, last):
    """(source, mode, normal, offset, pivot, xform, targets) of the real jobs; ``last`` = the pool's last slot."""
    if which == 0:
        return (0, _lib.MODE_SEQ, Z, 2.0, np.array([0, 0, 2], np.float32), _xforms(10, _lib.MODE_SEQ),
                [0, 1, S31, last, EMPTY, 2])
    if which == 1:
        return (S31, _lib.MODE_COMPOSED, N1, 2.2, np.array([0.05, 0.0, 2.2], np.float32),
                _xforms(11, _lib.MODE_COMPOSED), [S31, S31 - 1, S31 + 1, 0, last])
    return (last, _lib.MODE_TRANSLATE, Z, 2.0, np.zeros(3, np.float32), _xforms(12, _lib.MODE_TRANSLATE),
            [last, last - 1, S31, 0, EMPTY])


_proj_cache: dict = {}


def _oracle_proj(big, spec):
    key = (spec[0], spec[1])
    if key not in _proj_cache:
        cfg = big.cfg
        _proj_cache[key] = c_oracle.project(cfg.K_inv(), cfg.focal_length, cfg.cx, cfg.cy, H, W, big.packed[spec[0]],
                                            spec[2], spec[3], spec[4], spec[1], spec[5])
    return _proj_cache[key]


def _filler(n_cand, targets, source=EMPTY):
    return (source, _lib.MODE_SEQ, Z, 2.0, np.array([0, 0, 2], np.float32), _identity(n_cand), targets)


def _pass_case(big, size):
    """Jobs of the pass on the narrow or wide pool: real jobs at candidate slots 0, around S31 and at the end (around
    S32 on the wide pool), fillers of empty masks in between.  Returns (pool, specs, kinds, want projections)."""
    pool = big.narrow if size == "narrow" else big.wide
    last = len(pool) - 1
    n_total = N_NARROW if size == "narrow" else S32 - K_STRADDLE + N_REAL
    end = N_NARROW - N_REAL if size == "narrow" else S32 - K_STRADDLE
    real = [_real_spec(i, last) for i in range(3)]
    specs, kinds = [], []
    for kind, i, b, n in filler_layout(n_total, [(0, N_REAL), (S31 - K_STRADDLE, N_REAL), (end, N_REAL)]):
        specs.append(real[i] if kind == "real" else _filler(n, [EMPTY]))
        kinds.append(kind)
    want = [_oracle_proj(big, s) if k == "real" else None for s, k in zip(specs, kinds)]
    # the projections in the straddling slots have pixels on both sides of the boundary word
    reals = [i for i, k in enumerate(kinds) if k == "real"]
    assert _straddles(want[reals[1]][K_STRADDLE].reshape(-1), (1 << 31) - S31 * WORDS)
    if size == "wide":
        assert _straddles(want[reals[2]][K_STRADDLE].reshape(-1), (1 << 32) - S32 * WORDS)
    return pool, specs, kinds, want


def _check_pass(big, res, batch, kinds, want):
    """Real jobs against the oracle, exactly (only their slots are read); fillers: empty projections, zero table
    entries and the empty target's arg-max (candidate 0, 0 / 0 = NaN)."""
    popc_all, bbox_all = res.proj_popc.cpu().numpy(), res.proj_bbox.cpu().numpy()
    out = [t.cpu().numpy() for t in (res.best_cand, res.best_inter, res.best_union, res.best_iou)]
    for j, (jb, kind) in enumerate(zip(batch.jobs, kinds)):
        A, T = int(jb["n_cand"]), int(jb["n_tgt"])
        c0, t0, b0 = int(jb["cand_begin"]), int(jb["tgt_begin"]), int(jb["tab_begin"])
        sl = slice(t0, t0 + T)
        if kind == "filler":
            assert not popc_all[c0:c0 + A].any(), j
            assert (bbox_all[c0:c0 + A] == [0, -1, 0, -1]).all(), j
            assert _all_zero(res.proj_bits[c0:c0 + A]), f"filler job {j}: projected words not zero"
            assert _all_zero(res.inter_tab[b0:b0 + T * A], 1 << 28), f"filler job {j}: intersections not zero"
            assert not out[0][sl].any() and not out[1][sl].any() and not out[2][sl].any(), j
            assert np.isnan(out[3][sl]).all(), j
            continue
        proj = want[j]
        got = res.proj_bits[c0:c0 + A].cpu().numpy().view(np.uint32)
        diff = int(np.count_nonzero(got != proj))
        assert diff == 0, f"job {j} (slots {c0}..{c0 + A - 1}): {diff} projected words differ"
        assert np.array_equal(popc_all[c0:c0 + A], np.unpackbits(proj.view(np.uint8), axis=None).reshape(A, -1).sum(1))
        assert bbox_all[c0:c0 + A].tolist() == [_bbox_words(p) for p in proj], j
        inter, uni, best, iou = c_oracle.score(H, W, _packed(big, batch.tgt_index[sl]), proj)
        tab = res.inter_tab[b0:b0 + T * A].cpu().numpy()
        bad = int(np.count_nonzero(tab.reshape(T, A) != inter))
        assert bad == 0, f"job {j}: {bad} intersections differ"
        assert np.array_equal(out[0][sl], best), j
        assert np.array_equal(out[1][sl], inter[np.arange(T), best]), j
        assert np.array_equal(out[2][sl], uni[np.arange(T), best]), j
        nan = np.isnan(iou)
        assert np.array_equal(np.isnan(out[3][sl]), nan), j
        assert np.array_equal(out[3][sl][~nan].view(np.uint32), iou[~nan].view(np.uint32)), j


def _bbox_words(w: np.ndarray):
    if not w.any():
        return [0, -1, 0, -1]
    rows = np.where(w.any(1))[0]
    cols = np.where(w.any(0))[0]
    return [rows[0], rows[-1], cols[0], cols[-1]]


def _set_env(monkeypatch, **env):
    for k, v in env.items():
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)


# (scoring kernel, candidates per warp, arg-max key, projection kernel, projection schedule, output mode): every
# value of each appears on both pool sizes
PASS_CASES = [
    ("auto", None, "packed", "filter", "cta", "full"),
    ("ldg", "2", "wide", "exact", "persistent", "rows"),
    ("ldg", "4", "packed", "exact", "cta", "rows"),
    ("mma", None, "wide", "filter", "persistent", "full"),
    ("tma", None, "packed", "filter", "cta", "rows"),
]


@gpu
@pytest.mark.parametrize("case", PASS_CASES, ids=lambda c: "-".join(x for x in c if x))
@pytest.mark.parametrize("size", ["narrow", "wide"])
def test_pass_matches_oracle_across_2_31_and_2_32(big, size, case, monkeypatch):
    kernel, wc, key, proj, sched, out = case
    _set_env(monkeypatch, A3D_SCORE_KERNEL=None if kernel == "auto" else kernel, A3D_SCORE_WC=wc,
             A3D_SCORE_KEY="wide" if key == "wide" else None, A3D_SCORE_ADDR=None, A3D_PROJECT_KERNEL=proj,
             A3D_PROJECT_SCHED=sched, A3D_WS_POISON="1", A3D_TILE_PLAN=None, A3D_PASS_API=None)
    pool, specs, kinds, want = _pass_case(big, size)
    batch = engine.build_batch(*zip(*specs), pool.source_points)
    nc = len(batch.xform)
    assert (nc * WORDS < 1 << 32) == (size == "narrow") and (len(pool) * WORDS < 1 << 32) == (size == "narrow")
    _need(nc * WORDS * 4)
    res = engine.run_pass(big.cfg, pool, engine.DeviceBatch(batch, DEV), engine.Workspace(DEV), want_table=True,
                          out_mode=_lib.OUT_FULL if out == "full" else _lib.OUT_BBOX_ROWS)
    torch.cuda.synchronize()
    _check_pass(big, res, batch, kinds, want)


# ---------------------------------------------------------------------------------------------------------------
# 2. an intersection table past 2^31 entries
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kernel", ["ldg", "mma", "tma"])
def test_table_past_2_31_entries(big, kernel, monkeypatch):
    _set_env(monkeypatch, A3D_SCORE_KERNEL=kernel, A3D_SCORE_WC=None, A3D_SCORE_KEY=None, A3D_SCORE_ADDR=None,
             A3D_PROJECT_KERNEL=None, A3D_PROJECT_SCHED=None, A3D_WS_POISON="1", A3D_TILE_PLAN=None,
             A3D_PASS_API=None)
    n_fill = table_filler_targets(4096, 1 << 31)
    real = _real_spec(1, S32)
    real = real[:6] + ([S31, S31 - 1, S31 + 1, 0, S32, S32 - 1, EMPTY, 2] * 3,)
    specs = [_filler(4096, np.full(n_fill, EMPTY, np.int32)), real]
    batch = engine.build_batch(*zip(*specs), big.wide.source_points)
    tab_begin = int(batch.jobs["tab_begin"][1])
    assert tab_begin < 1 << 31 < tab_begin + 24 * N_REAL
    _need((tab_begin + 24 * N_REAL) * 4)
    res = engine.run_pass(big.cfg, big.wide, engine.DeviceBatch(batch, DEV), engine.Workspace(DEV), want_table=True)
    torch.cuda.synchronize()
    _check_pass(big, res, batch, ["filler", "real"], [None, _oracle_proj(big, real)])


# ---------------------------------------------------------------------------------------------------------------
# 3. a point-cloud workspace past 2^31 floats
# ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("proj", ["exact", "filter"])
def test_point_cloud_workspace_past_2_31_floats(big, proj, monkeypatch):
    _set_env(monkeypatch, A3D_SCORE_KERNEL=None, A3D_SCORE_WC=None, A3D_SCORE_KEY=None, A3D_SCORE_ADDR=None,
             A3D_PROJECT_KERNEL=proj, A3D_PROJECT_SCHED=None, A3D_WS_POISON="1", A3D_TILE_PLAN=None,
             A3D_PASS_API=None)
    n_fill = pcd_fillers(H * W, _lib.PCD_PLANES, 1 << 31)
    real = _real_spec(1, S32)
    specs = [_filler(1, [EMPTY], source=FULL)] * n_fill + [real]
    batch = engine.build_batch(*zip(*specs), big.wide.source_points)
    assert int(batch.jobs["pcd_cap"][0]) == H * W
    pcd_begin = int(batch.jobs["pcd_begin"][-1])
    assert _lib.PCD_PLANES * pcd_begin > 1 << 31
    _need(_lib.PCD_PLANES * (pcd_begin + H * W) * 4)
    res = engine.run_pass(big.cfg, big.wide, engine.DeviceBatch(batch, DEV), engine.Workspace(DEV), want_table=True)
    torch.cuda.synchronize()
    want_real = _oracle_proj(big, real)
    # the fillers project a full frame onto an empty target: only their scores are checked (candidate 0, nothing in
    # common, the union is the candidate's pixel count, IoU 0)
    out = [t.cpu().numpy() for t in (res.best_cand, res.best_inter, res.best_union, res.best_iou)]
    popc = res.proj_popc[:n_fill].cpu().numpy()
    assert (popc > 0).all() and np.array_equal(out[2][:n_fill], popc)
    assert not out[0][:n_fill].any() and not out[1][:n_fill].any() and not out[3][:n_fill].any()
    last = batch.jobs[-1:]
    _check_pass(big, res, SimpleNamespace(jobs=last, tgt_index=batch.tgt_index), ["real"], [want_real])


# ---------------------------------------------------------------------------------------------------------------
# 4. per-mask kernels on the 447,393-mask pool
# ---------------------------------------------------------------------------------------------------------------
def _bbox_pixels(m: np.ndarray):
    if not m.any():
        return [0, -1, 0, -1]
    rows = np.flatnonzero(m.any(1))
    cols = np.flatnonzero(m.any(0))
    return [rows[0], rows[-1], cols[0] // 32, cols[-1] // 32]


@gpu
def test_mask_meta_of_every_slot(big):
    pool = engine.pool_from_bits(big.bits, H, W)
    popc, bbox = pool.popc.cpu().numpy(), pool.bbox.cpu().numpy()
    want_popc = np.zeros(N_WIDE, np.int64)
    want_bbox = np.tile(np.array([0, -1, 0, -1]), (N_WIDE, 1))
    for s, m in big.masks.items():
        want_popc[s] = m.sum()
        want_bbox[s] = _bbox_pixels(m)
    assert np.array_equal(popc, want_popc)
    bad = np.flatnonzero((bbox != want_bbox).any(1))
    assert bad.size == 0, f"boxes differ at slots {bad[:8].tolist()}"


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.uint8], ids=["f32", "u8"])
def test_emit_far_masks(big, dtype):
    idx = torch.tensor(FAR + [EMPTY, 0], dtype=torch.int32, device=DEV)
    got = engine.emit_masks(big.bits, idx, H, W, dtype).cpu().numpy()
    assert np.array_equal(got, _dense(big, FAR + [EMPTY, 0]).astype(got.dtype))
    # one contiguous call of the pool's last 7,000 masks: more than 2^31 output elements, the placed ones at its end
    n = 7000
    _need(n * H * W * torch.tensor([], dtype=dtype).element_size())
    out = engine.emit_masks(big.bits[N_WIDE - n:], None, H, W, dtype)
    first = F32_FRAME
    assert N_WIDE - n + first == S32 - 9 and (first + 1) * H * W > 1 << 31 > first * H * W
    tail = out[first:].cpu().numpy()
    assert np.array_equal(tail, _dense(big, range(S32 - 9, S32 + 1)).astype(tail.dtype))
    assert _all_zero(out[:first], 512)


@gpu
def test_bits_to_rle_of_far_masks(big):
    sel = FAR + [EMPTY, FULL]
    counts, begin = engine.bits_to_rle(big.bits, H, W, index=torch.tensor(sel, dtype=torch.int32))
    for i, s in enumerate(sel):
        want = rle.rle_counts(rle.encode(big.masks.get(s, np.zeros((H, W), bool))))
        assert np.array_equal(counts[begin[i]:begin[i + 1]], want), s


@gpu
def test_rle_to_bits_past_2_31_words(big):
    n = 224_000
    assert n * WORDS > 1 << 31 and S31 + 1 < n
    placed = {s: rle.rle_counts(rle.encode(m)) for s, m in big.masks.items() if s < n}
    assert S31 in placed and FULL in placed
    counts, begin = rle_call_arrays(n, H * W, placed)
    _need(n * WORDS * 4)
    lib = _lib.load()
    out = torch.full((n, H, PITCH), -0x54545455, dtype=torch.int32, device=DEV)      # 0xAB bytes
    d_counts = torch.from_numpy(counts.view(np.int32)).to(DEV)
    d_begin = torch.from_numpy(begin).to(DEV)
    _lib.check(lib.a3d_rle_to_bits(d_counts.data_ptr(), d_begin.data_ptr(), n, H, W, out.data_ptr(),
                                   engine._stream_ptr()), "a3d_rle_to_bits")
    idx = torch.tensor(sorted(placed), device=DEV)
    assert torch.equal(out.index_select(0, idx), big.bits.index_select(0, idx))
    popc, _ = engine.mask_meta(out, H, W)
    assert int(popc.sum(dtype=torch.int64)) == sum(int(big.masks[s].sum()) for s in placed)


@gpu
def test_upload_masks_past_2_32_words(big):
    k, reps = 1024, 437
    n = k * reps
    assert n * WORDS > 1 << 32
    _need(n * WORDS * 4 + k * H * W)
    rng = np.random.RandomState(4)
    sel = [big.masks[s] for s in PLACED]
    chunk = np.stack([sel[i % len(sel)] for i in range(k)]).astype(np.uint8)
    chunk[np.arange(k), rng.randint(0, H, k), rng.randint(0, W, k)] ^= 1            # every mask of the chunk differs
    host = torch.from_numpy(chunk).pin_memory()
    want = engine.pack_masks(torch.from_numpy(chunk).to(DEV)).bits
    bits = torch.full((n, H, PITCH), -0x54545455, dtype=torch.int32, device=DEV)
    stage = torch.empty(k, H, W, dtype=torch.uint8, device=DEV)
    ptrs = (C.c_void_p * reps)(*([host.data_ptr()] * reps))
    cnt = (C.c_int64 * reps)(*([k] * reps))
    _lib.check(_lib.load().a3d_upload_masks(ptrs, cnt, reps, _lib.A3D_U8, H, W, 0.5, stage.data_ptr(), k,
                                            bits.data_ptr(), None, 4, engine._stream_ptr()), "a3d_upload_masks")
    torch.cuda.synchronize()
    bad = [b for b in range(reps) if not torch.equal(bits[b * k:(b + 1) * k], want)]
    assert not bad, f"blocks {bad[:8]} of {reps} differ"


# ---------------------------------------------------------------------------------------------------------------
# 5. frame-indexed kernels past 2^31 elements
# ---------------------------------------------------------------------------------------------------------------
def _compact(slots):
    """Mask slots -> (sorted unique slots, index of every slot in them)."""
    u = sorted(set(int(s) for s in slots))
    return u, np.array([u.index(int(s)) for s in slots], np.int64)


@gpu
def test_plane_offsets_past_2_31_depth_floats(big):
    F = 7000
    assert F * H * W > 1 << 31
    _need(F * H * W * 4)
    depth = torch.empty(F, H, W, dtype=torch.float32, device=DEV)
    yy, xx = torch.meshgrid(torch.arange(H, device=DEV, dtype=torch.float32),
                            torch.arange(W, device=DEV, dtype=torch.float32), indexing="ij")
    base = 1.5 + yy / 512 + xx / 1024
    for a in range(0, F, 500):
        f = torch.arange(a, min(F, a + 500), device=DEV, dtype=torch.float32)
        depth[a:a + 500] = base[None] + (f % 97)[:, None, None] / 64
    kinv = big.cfg.K_inv().astype(np.float32)
    x, y = np.meshgrid(np.arange(W, dtype=np.float32), np.arange(H, dtype=np.float32))
    rays = np.stack([kinv[0, 0] * x + kinv[0, 2], kinv[1, 1] * y + kinv[1, 2], np.ones_like(x)]).astype(np.float32)
    inst_mask = np.array([S32, S31, S32 - 1, 0, S31 + 1, S32, FULL, EMPTY], np.int32)
    inst_frame = np.array([F32_FRAME, F32_FRAME, F - 1, 0, F - 1, 0, F32_FRAME, F - 1], np.int32)
    normals = np.random.RandomState(6).randn(len(inst_mask), 3).astype(np.float32)
    off, cnt = engine.plane_offsets(big.wide, torch.from_numpy(inst_mask).to(DEV), torch.from_numpy(normals).to(DEV),
                                    torch.from_numpy(rays).to(DEV), depth, torch.from_numpy(inst_frame).to(DEV))
    torch.cuda.synchronize()
    mslots, mi = _compact(inst_mask)
    fr, fi = _compact(inst_frame)
    dframes = depth.index_select(0, torch.tensor(fr, device=DEV)).cpu().numpy()
    want = reference(_dense(big, mslots), mi, normals, rays, dframes, fi)
    assert want[1][-1] == 0 and want[1][-2] == H * W
    assert_offsets(off, cnt, want, "large offsets")


@gpu
def test_render_past_2_31_bytes(big):
    F = 2400
    assert (RGB_FRAME + 1) * H * W * 3 > 1 << 31 and F * H * W * 3 > 1 << 31
    _need(2 * F * H * W * 3)
    bg = torch.empty(F, H, W, 3, dtype=torch.uint8, device=DEV)
    yy, xx = torch.meshgrid(torch.arange(H, device=DEV), torch.arange(W, device=DEV), indexing="ij")
    base = torch.stack([yy + xx, 3 * yy + xx // 2, xx * 5 + yy // 3], -1).to(torch.int32)
    for a in range(0, F, 200):
        f = torch.arange(a, min(F, a + 200), device=DEV, dtype=torch.int32)
        bg[a:a + 200] = ((base[None] + 7 * f[:, None, None, None]) % 256).to(torch.uint8)
    lay = {RGB_FRAME: [(S32, _lib.LAYER_FILL, (200, 30, 40, 128)), (S31, _lib.LAYER_OUTLINE, (10, 250, 10, 255)),
                       (S32 - 1, _lib.LAYER_FILL, (0, 0, 255, 60))],
           F - 3: [(S31, _lib.LAYER_FILL, (255, 255, 0, 255))],
           F - 1: [(S32, _lib.LAYER_OUTLINE, (1, 2, 3, 200)), (S32 - 2, _lib.LAYER_FILL, (90, 80, 70, 254))]}
    checked = [RGB_FRAME, F - 3, F - 2, F - 1]
    rows = [r for f in range(F) for r in lay.get(f, [])]
    lb = np.concatenate(([0], np.cumsum([len(lay.get(f, [])) for f in range(F)])))
    layers = np.array(rows, dtype=_lib.LAYER_DTYPE)
    segs = np.zeros(0, _lib.SEGMENT_DTYPE)
    out = engine.render(big.wide, layers, lb, segs, np.zeros(F + 1, np.int64), bg)
    torch.cuda.synchronize()
    mslots, mi = _compact(layers["mask"])
    cl = layers.copy()
    cl["mask"] = mi
    clb = np.concatenate(([0], np.cumsum([len(lay.get(f, [])) for f in checked])))
    # the checked frames' layers, in frame order, are all the layers
    assert np.array_equal(np.concatenate([layers[lb[f]:lb[f + 1]] for f in checked]), layers)
    idx = torch.tensor(checked, device=DEV)
    want = render_ref.composite(bg.index_select(0, idx).cpu().numpy(), _dense(big, mslots), cl, clb, segs,
                                np.zeros(len(checked) + 1, np.int64))
    got = out.index_select(0, idx).cpu().numpy()
    bad = np.argwhere(got != want)
    assert len(bad) == 0, f"{len(bad)} bytes differ, first at {bad[:5].tolist()} (frames {checked})"
    assert not np.array_equal(got[0], bg[RGB_FRAME].cpu().numpy())
    for a, b in ((0, RGB_FRAME), (RGB_FRAME + 1, F - 3)):
        for c in range(a, b, 256):
            assert torch.equal(out[c:min(b, c + 256)], bg[c:min(b, c + 256)]), f"frames {c}.. differ from the background"


@gpu
def test_plane_maps_past_2_31_elements(big):
    F = 7000
    assert (RGB_FRAME + 1) * H * W * 3 > 1 << 31 and (F32_FRAME + 1) * H * W > 1 << 31
    _need(F * H * W * 7)
    bg_rgb = (12, 34, 56)

    def n(v):
        v = np.asarray(v, np.float64)
        return tuple((v / np.linalg.norm(v)).astype(np.float32))

    lay = {RGB_FRAME: [(S32, n([0.1, 0.0, 1.0]), 2.0, (250, 0, 0)), (S31, n([-0.2, 0.1, 1.0]), 2.1, (0, 250, 0))],
           F32_FRAME: [(S31, n([0.0, 0.3, 1.0]), 1.8, (0, 0, 250)), (S32 - 1, Z, 1.9, (9, 99, 199))],
           F - 1: [(S32, Z, 2.5, (77, 88, 99)), (FULL, n([0.05, -0.05, 1.0]), 3.0, (1, 1, 1))]}
    checked = [RGB_FRAME, F32_FRAME, F - 1]
    rows = [(m, nv, off, rgb, 0) for f in range(F) for (m, nv, off, rgb) in lay.get(f, [])]
    lb = np.concatenate(([0], np.cumsum([len(lay.get(f, [])) for f in range(F)])))
    layers = np.array(rows, dtype=_lib.PLANE_LAYER_DTYPE)
    depth, rgb = engine.plane_maps(big.wide, layers, lb, big.cfg, bg_rgb)
    torch.cuda.synchronize()
    mslots, mi = _compact(layers["mask"])
    cl = layers.copy()
    cl["mask"] = mi
    clb = np.concatenate(([0], np.cumsum([len(lay[f]) for f in checked])))
    wd, wr = plane_maps_ref.plane_maps(big.cfg.K_inv(), _dense(big, mslots), cl, clb, bg_rgb)
    idx = torch.tensor(checked, device=DEV)
    gd, gr = depth.index_select(0, idx).cpu().numpy(), rgb.index_select(0, idx).cpu().numpy()
    bad = np.argwhere(gd.view(np.int32) != wd.view(np.int32))
    assert len(bad) == 0, f"{len(bad)} depths differ, first at {bad[:5].tolist()} (frames {checked})"
    bad = np.argwhere(gr != wr)
    assert len(bad) == 0, f"{len(bad)} colour bytes differ, first at {bad[:5].tolist()} (frames {checked})"
    assert (wd > 0).any(axis=(1, 2)).all()
    bgc = torch.tensor(bg_rgb, dtype=torch.uint8, device=DEV)
    for a, b in ((0, RGB_FRAME), (RGB_FRAME + 1, F32_FRAME), (F32_FRAME + 1, F - 1)):
        for c in range(a, b, 256):
            e = min(b, c + 256)
            assert _all_zero(depth[c:e], 64), f"frames {c}..{e - 1}: depth not 0"
            assert bool((rgb[c:e] == bgc).all()), f"frames {c}..{e - 1}: colour not the background"
