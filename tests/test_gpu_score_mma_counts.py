"""k_score_mma at counts large enough to expose a short accumulator.

The tensor-core scoring kernel contracts masks expanded to e2m1 nibbles (0 or 1.0) into f32 accumulators in
tensor memory, which hold every count up to 2^24 exactly.  These cases force it (A3D_SCORE_KERNEL=mma) on whole
frames of ones, a checkerboard against its complement, random dense masks whose counts straddle 2^14, 2^16 and
2^20, regions of an odd number of word positions (the last MMA pairs a position with zeros) and 16, 192 and 240
candidates per tile, and compare inter, union, arg-max and the IoU bits with a numpy popcount reference.  Frames
over 2^24 pixels must be scored exactly too: the library takes k_score for them even when mma is asked for."""
import numpy as np
import pytest
import torch

from articulation3d_b200 import _lib, engine

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(autouse=True)
def mma_kernel(monkeypatch):
    monkeypatch.setenv("A3D_SCORE_KERNEL", "mma")
    monkeypatch.delenv("A3D_SCORE_KEY", raising=False)


def _masks(H, W, density, seed, box=None):
    """(n, H, W) bool masks on the device, mask i dense at density[i] (1.0 = all ones), optionally confined to
    box = (r0, r1, c0, c1) (inclusive)."""
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    d = torch.tensor(density, dtype=torch.float32, device=DEV)
    m = torch.rand((len(density), H, W), generator=g, device=DEV) < d[:, None, None]
    if box is not None:
        r0, r1, c0, c1 = box
        keep = torch.zeros((H, W), dtype=torch.bool, device=DEV)
        keep[r0:r1 + 1, c0:c1 + 1] = True
        m &= keep
    return m


def _score(H, W, tgt, cand):
    """a3d_score of one job (every target against every candidate) -> (best rows, inter table)."""
    lib = _lib.load()
    tp, cp = engine.pack_masks(tgt), engine.pack_masks(cand)
    T, N = len(tgt), len(cand)
    jobs = np.zeros(1, _lib.JOB_DTYPE)
    jobs[0]["n_cand"], jobs[0]["n_tgt"] = N, T
    d_jobs = torch.from_numpy(jobs.view(np.uint8).copy()).to(DEV)
    d_tidx = torch.arange(T, dtype=torch.int32, device=DEV)
    key_ws = torch.full((T,), -1, dtype=torch.int64, device=DEV)
    inter_tab = torch.full((T * N,), -7, dtype=torch.int32, device=DEV)
    out = torch.full((4, T), -7, dtype=torch.int32, device=DEV)
    _lib.check(lib.a3d_score(H, W, d_jobs.data_ptr(), 1, T, N, T, T, N, tp.bits.data_ptr(), tp.popc.data_ptr(),
                             tp.bbox.data_ptr(), d_tidx.data_ptr(), cp.bits.data_ptr(), cp.popc.data_ptr(),
                             cp.bbox.data_ptr(), key_ws.data_ptr(), inter_tab.data_ptr(), out[0].data_ptr(),
                             out[1].data_ptr(), out[2].data_ptr(), out[3].data_ptr(), engine._stream_ptr()),
               "a3d_score")
    torch.cuda.synchronize()
    tb = tp.bits.view(T, -1).cpu().numpy().view(np.uint32)
    cb = cp.bits.view(N, -1).cpu().numpy().view(np.uint32)
    return out.cpu().numpy(), inter_tab.cpu().numpy().reshape(T, N), tb, cb


def _check(out, tab, tb, cb):
    """numpy popcount reference: int64 inter / union, fp32 divide, first maximum.  Returns inter."""
    inter = np.stack([np.bitwise_count(t & cb).sum(1, dtype=np.int64) for t in tb])
    union = (np.bitwise_count(tb).sum(1, dtype=np.int64)[:, None] + np.bitwise_count(cb).sum(1, dtype=np.int64)[None, :]
             - inter)
    assert np.array_equal(tab, inter)
    iou = inter.astype(np.float32) / union.astype(np.float32)       # correctly rounded, as __fdiv_rn
    best = iou.argmax(1)
    rows = np.arange(len(tb))
    assert np.array_equal(out[0], best)
    assert np.array_equal(out[1], inter[rows, best])
    assert np.array_equal(out[2], union[rows, best])
    assert np.array_equal(out[3].view(np.float32).view(np.uint32), iou[rows, best].view(np.uint32))
    return inter


@pytest.mark.parametrize("n_cand", [16, 192, 240])
@pytest.mark.parametrize("H,W", [(480, 640), (768, 1024)])
def test_full_frame_all_ones(H, W, n_cand):
    """inter = H * W in every accumulator, ties everywhere (the first candidate wins)."""
    tgt = torch.ones((128, H, W), dtype=torch.bool, device=DEV)
    cand = torch.ones((n_cand, H, W), dtype=torch.bool, device=DEV)
    out, tab, tb, cb = _score(H, W, tgt, cand)
    inter = _check(out, tab, tb, cb)
    assert (inter == H * W).all()


@pytest.mark.parametrize("n_cand", [16, 240])
def test_checkerboard_against_complement(n_cand):
    """Every pixel of the frame meets a zero: inter = 0 over 768 x 1024."""
    H, W = 768, 1024
    yy, xx = torch.meshgrid(torch.arange(H, device=DEV), torch.arange(W, device=DEV), indexing="ij")
    board = (yy + xx) % 2 == 0
    tgt = board.expand(64, H, W).contiguous()
    cand = (~board).expand(n_cand, H, W).contiguous()
    out, tab, tb, cb = _score(H, W, tgt, cand)
    inter = _check(out, tab, tb, cb)
    assert (inter == 0).all()


@pytest.mark.parametrize("n_cand", [16, 192, 240])
def test_random_dense_counts_straddle_powers_of_two(n_cand):
    """1024 x 1280 frames (2^20 pixels and more: the wide arg-max key), densities from 2 % to all ones."""
    H, W = 1024, 1280
    tgt = _masks(H, W, [(0.02, 0.1, 0.5, 0.95, 1.0)[i % 5] for i in range(64)], 1 + n_cand)
    cand = _masks(H, W, [(0.5, 0.8, 0.95, 1.0, 0.03, 0.012)[i % 6] for i in range(n_cand)], 2 + n_cand)
    out, tab, tb, cb = _score(H, W, tgt, cand)
    inter = _check(out, tab, tb, cb)
    for p in (14, 16, 20):
        assert (inter < 2 ** p).any() and (inter > 2 ** p).any(), p


@pytest.mark.parametrize("n_cand", [16, 192, 240])
@pytest.mark.parametrize("H,W,box", [(481, 672, None), (480, 640, (17, 317, 64, 287))])
def test_odd_word_position_count(H, W, box, n_cand):
    """Regions of 481 x 21 and 301 x 7 word positions: the last MMA reads one position and a zero chunk."""
    tgt = _masks(H, W, [(0.7, 1.0, 0.3)[i % 3] for i in range(96)], 3 + n_cand, box)
    cand = _masks(H, W, [(0.6, 1.0, 0.9, 0.2)[i % 4] for i in range(n_cand)], 4 + n_cand, box)
    out, tab, tb, cb = _score(H, W, tgt, cand)
    _check(out, tab, tb, cb)


def test_frames_over_2_24_pixels_are_scored_exactly():
    """4097 x 4096 frames: odd counts above 2^24 have no f32 representation, so the library scores them on
    the integer pipes although mma is asked for."""
    H, W = 4097, 4096
    tgt = torch.ones((2, H, W), dtype=torch.bool, device=DEV)
    tgt[1, 5, 7] = False
    cand = torch.ones((3, H, W), dtype=torch.bool, device=DEV)
    cand[0, 4000, 4095] = False
    cand[2] = _masks(H, W, [0.5], 5)[0]
    out, tab, tb, cb = _score(H, W, tgt, cand)
    inter = _check(out, tab, tb, cb)
    assert inter[0, 0] == H * W - 1 and inter[1, 1] == H * W - 1 and inter[1, 0] == H * W - 2
