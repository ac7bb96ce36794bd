"""CPU tests of the library's COCO RLE string writer (a3d_host_rle_strings) against rle.counts_to_string."""
import numpy as np
import pytest

from articulation3d_b200 import _lib, rle


def _masks():
    """The masks of test_native_string_decoder_equals_python_decoder."""
    rng = np.random.RandomState(3)
    H, W = 120, 160
    masks = []
    m = np.zeros((H, W), bool); masks.append(m.copy())
    m[:] = True; masks.append(m.copy())
    m[:] = False; m[20:90, 30:100] = True; masks.append(m.copy())
    masks.append(rng.rand(H, W) < 0.5)
    masks.append(rng.rand(H, W) < 0.01)
    m = np.zeros((H, W), bool); m[0, 0] = m[-1, -1] = True; masks.append(m.copy())
    m = np.zeros((H, W), bool); m[:, ::2] = True; masks.append(m.copy())
    return masks


def _random_count_lists():
    rng = np.random.RandomState(11)
    lists = [[0], [5], [2 ** 32 - 1], [], [0, 0, 0, 0], [0, 2 ** 32 - 1, 0, 2 ** 32 - 1, 0, 1]]
    lists.append([2 ** 31 - 1, 1, 0, 2 ** 31, 2 ** 32 - 1, 0, 7])           # deltas of both signs across int32
    for k in range(40):
        n = rng.randint(1, 60)
        hi = [16, 1 << 15, 1 << 20, (1 << 21) + 5, 1 << 31, 1 << 32][k % 6]
        c = rng.randint(0, hi, size=n, dtype=np.int64)
        c[rng.rand(n) < 0.2] = 0
        lists.append(c.tolist())
    return lists


def test_host_strings_equal_python_writer_and_round_trip():
    count_lists = [rle.rle_counts(rle.encode(m)).tolist() for m in _masks()] + _random_count_lists()
    begin = np.zeros(len(count_lists) + 1, np.int64)
    begin[1:] = np.cumsum([len(c) for c in count_lists])
    flat = np.array([x for c in count_lists for x in c], dtype=np.uint32)
    got = rle.counts_to_strings(flat, begin)
    assert len(got) == len(count_lists)
    for c, s in zip(count_lists, got):
        assert isinstance(s, bytes) and s == rle.counts_to_string(c), c
    # back through the library's decoder
    back, cbeg, _ = rle.strings_to_counts(got)
    assert np.array_equal(back, flat) and np.array_equal(cbeg, begin)


def test_host_strings_single_count_and_no_masks():
    assert rle.counts_to_strings(np.array([307200], np.uint32), np.array([0, 1])) == [rle.counts_to_string([307200])]
    assert rle.counts_to_strings(np.zeros(0, np.uint32), np.array([0, 0])) == [b""]
    assert rle.counts_to_strings(np.zeros(0, np.uint32), np.array([0])) == []


def test_host_strings_refuses_small_buffer_and_bad_offsets():
    lib = _lib.load()
    counts = np.array([100000, 3, 2 ** 32 - 1, 0], np.uint32)
    begin = np.array([0, 4], np.int64)
    need = len(rle.counts_to_string(counts))
    chars = np.full(need + 8, 0xAB, np.uint8)
    cbeg = np.zeros(2, np.int64)
    assert lib.a3d_host_rle_strings(counts.ctypes.data, begin.ctypes.data, 1, chars.ctypes.data, need,
                                    cbeg.ctypes.data) == need
    assert chars[:need].tobytes() == rle.counts_to_string(counts) and np.all(chars[need:] == 0xAB)
    assert cbeg.tolist() == [0, need]
    rc = lib.a3d_host_rle_strings(counts.ctypes.data, begin.ctypes.data, 1, chars.ctypes.data, need - 1,
                                  cbeg.ctypes.data)
    assert rc == -1 and b"more are needed" in lib.a3d_last_error_string()
    bad = np.array([2, 1], np.int64)
    assert lib.a3d_host_rle_strings(counts.ctypes.data, bad.ctypes.data, 1, chars.ctypes.data, need, None) == -1
    assert lib.a3d_host_rle_strings(None, None, -1, None, 0, None) == -1


@pytest.mark.parametrize("shape", [(1, 1), (5, 7), (33, 100)])
def test_encode_many_without_device_is_encode(shape):
    rng = np.random.RandomState(shape[1])
    masks = (rng.rand(4, *shape) < 0.3).astype(np.float32)
    assert rle.encode_many(masks) == [rle.encode(m) for m in masks]
