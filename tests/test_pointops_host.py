"""Segment FPS / kNN of packed variable-size clouds, host side: the fp32 oracle (oracle/pdae_oracle_pointops.c) against
float64 transcriptions of the published pointops loops -- the literal block tree and the literal per-thread heap --,
the padding of short, empty and uncovered segments, and argument rejection by the C ABI without a GPU."""
import numpy as np
import pytest

from oracle import cpu_pointops as cp
from pointdae_b200 import _native

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3


def packed(sizes, seed, grid=None):
    """clouds of the given sizes back to back: uniform in the unit cube, or small-integer grid points (exact in fp32
    and float64, so distances tie)"""
    rng = np.random.default_rng(seed)
    n = int(sum(sizes))
    x = rng.integers(0, grid, (n, 3)) if grid else rng.random((n, 3))
    return x.astype(np.float32), np.cumsum(sizes).astype(np.int32)


def sample_offsets(sizes, frac, minimum=1):
    return np.cumsum([max(minimum, int(s * frac)) for s in sizes]).astype(np.int32)


@pytest.mark.parametrize("sizes,frac,n", [
    ([100, 0, 1, 300, 30], 0.2, None),
    ([1023, 5, 700], 0.05, None),          # bs 512
    ([1024, 3], 0.05, None),               # bs 1024
    ([1025, 900], 0.05, None),
    ([600, 1100, 40], 0.05, 200),          # n below the largest segment: bs from n, segments larger than n
])
def test_fps_oracle_matches_published_tree(sizes, frac, n):
    x, off = packed(sizes, 1)
    noff = sample_offsets(sizes, frac)
    n = cp.largest(off) if n is None else n
    idx, tmp = cp.seg_fps(x, off, noff, n=n, tmp=np.full(len(x), 1e10, np.float32))
    ref_idx, ref_tmp = cp.fps_published_f64(x, off, noff, n)
    assert np.array_equal(idx, ref_idx)
    assert np.allclose(tmp, ref_tmp, rtol=1e-6, atol=0)
    assert np.array_equal(cp.seg_fps(x, off, noff, n=n)[0], idx)  # tmp = null: same samples


@pytest.mark.parametrize("n", [7, 64, 1023, 1024])
def test_fps_tie_rule_on_grid(n):
    # integer grid points: float64 and fp32 distances are the same integers, so every tie is real and the two agree bit
    # for bit, minima included
    sizes = [300, 64, 0, 200]
    x, off = packed(sizes, 2, grid=4)
    noff = sample_offsets(sizes, 0.3)
    idx, tmp = cp.seg_fps(x, off, noff, n=n, tmp=np.full(len(x), 1e10, np.float32))
    ref_idx, ref_tmp = cp.fps_published_f64(x, off, noff, n)
    assert np.array_equal(idx, ref_idx)
    assert np.array_equal(tmp, ref_tmp.astype(np.float32))


def test_fps_padding_and_tmp():
    x, off = packed([5, 0, 3], 3)
    noff = np.array([2, 6, 6], np.int32)  # 4 samples of the empty segment, none for the last
    idx, _ = cp.seg_fps(x, off, noff)
    assert idx.tolist() == [0, idx[1], 5, 5, 5, 5]
    # tmp holds the minima folded with every sample but the last; a 1-sample segment leaves its tmp alone
    t0 = np.arange(8, dtype=np.float32) + 50.0
    _, t = cp.seg_fps(x, off, np.array([1, 1, 1], np.int32), tmp=t0)
    assert np.array_equal(t, t0)
    _, t = cp.seg_fps(x, off, np.array([2, 2, 2], np.int32), tmp=np.full(8, 1e10, np.float32))
    d = ((x[:5] - x[0]) ** 2).sum(-1)
    assert np.allclose(t[:5], d, rtol=1e-6) and (t[5:] == 1e10).all()


def _heap_equals_order_up_to_kth_ties(hi, hd, oi, od):
    """the published heap's row against the (d^2, index) order: the same distances; the same indices except among
    the entries tied with the k-th distance, which the heap may keep and order differently"""
    assert np.array_equal(hd, od)
    for r in range(hi.shape[0]):
        kth = od[r, -1]
        keep = od[r] != kth
        assert np.array_equal(oi[r, keep], hi[r, keep]) or np.array_equal(
            oi[r, keep], hi[r][np.lexsort((hi[r], hd[r]))][keep])


@pytest.mark.parametrize("sizes,nsample", [([100, 0, 1, 300, 30], 16), ([500, 20, 257], 100), ([64, 64], 1)])
def test_knn_oracle_matches_published_heap(sizes, nsample):
    x, off = packed(sizes, 4)
    idx, d2 = cp.seg_knn(nsample, x, x, off, off)
    ref_i, ref_d = cp.knn_published_f64(nsample, x, x, off, off)
    # random coordinates: no ties, so the literal heap and the defined order agree on every index
    assert np.array_equal(idx, ref_i)
    assert np.allclose(d2, ref_d, rtol=1e-6, atol=0)


def test_knn_ties_are_the_only_difference():
    sizes = [200, 90, 0, 150]
    x, off = packed(sizes, 5, grid=3)  # 27 distinct points: masses of exact ties
    q, qoff = packed([40, 40, 5, 40], 6, grid=3)
    idx, d2 = cp.seg_knn(20, x, q, off, qoff)
    hi, hd = cp.knn_published_f64(20, x, q, off, qoff)
    _heap_equals_order_up_to_kth_ties(hi, hd.astype(np.float32), idx, d2)
    # the defined order: ascending (d^2, index) within every row
    for r in range(len(q)):
        keys = list(zip(d2[r].tolist(), idx[r].tolist()))
        assert keys == sorted(keys)


def test_knn_padding():
    x, off = packed([5, 0, 3], 7)
    q = np.random.default_rng(8).random((9, 3)).astype(np.float32)
    qoff = np.array([3, 5, 7], np.int32)  # rows 7 and 8 lie past the last segment
    idx, d2 = cp.seg_knn(4, x, q, off, qoff)
    assert (d2[0:3] < 1e10).all()                                      # 5 points for 4 slots
    assert (idx[3:5] == 5).all() and (d2[3:5] == 1e10).all()          # empty segment: the heap's initial value
    assert (idx[5:7, 3] == 5) .all() and (d2[5:7, 3] == 1e10).all()   # 3 points for 4 slots
    assert set(idx[5].tolist()[:3]) == {5, 6, 7}
    assert (idx[7:] == -1).all() and (d2[7:] == 1e10).all()
    ref_i, ref_d = cp.knn_published_f64(4, x, q, off, qoff)
    assert np.array_equal(idx[:7], ref_i[:7]) and np.allclose(d2[:7], ref_d[:7], rtol=1e-6)
    # a distance of 1e10 or more never enters the heap
    far = np.array([[0, 0, 0], [1e6, 0, 0]], np.float32)
    i2, dd = cp.seg_knn(2, far, far[:1], np.array([2], np.int32), np.array([1], np.int32))
    assert i2.tolist() == [[0, 0]] and dd.tolist() == [[0.0, 1e10]]


def test_block_size_rule():
    assert [cp.block_size(v) for v in (0, 1, 2, 3, 511, 512, 1023, 1024, 1025, 5000)] == [
        1, 1, 2, 2, 256, 512, 512, 1024, 1024, 1024]


def test_abi_rejects_bad_arguments():
    L = _native.lib()
    fake = 256
    assert L.pdae_seg_fps_workspace_bytes(0) == 0
    assert L.pdae_seg_fps_workspace_bytes(1000) == 4096
    assert L.pdae_seg_knn_workspace_bytes(4, 100) == 256 + 256 * ((16 * (13 + 4) + 255) // 256)
    assert L.pdae_seg_knn_workspace_bytes(4, 0) == 0
    # fps(xyz, n_total, offset, new_offset, b, n, m_total, tmp, idx, ws, ws_bytes, stream)
    assert L.pdae_seg_fps_f32(None, 10, None, None, -1, 4, 4, None, None, None, 0, None) == E_INVALID
    assert L.pdae_seg_fps_f32(None, 10, None, None, 2, -4, 4, None, None, None, 0, None) == E_INVALID
    assert L.pdae_seg_fps_f32(None, 10, None, None, 0, 4, 4, None, None, None, 0, None) == 0      # no segments
    assert L.pdae_seg_fps_f32(None, 10, None, None, 2, 4, 0, None, None, None, 0, None) == 0      # no samples
    assert L.pdae_seg_fps_f32(None, 10, fake, fake, 2, 4, 4, None, fake, fake, 4096, None) == E_INVALID  # no xyz
    assert L.pdae_seg_fps_f32(fake, 10, fake, fake, 2, 4, 4, None, fake, None, 0, None) == E_WORKSPACE
    assert L.pdae_seg_fps_f32(fake, 1 << 22, fake, fake, 2, 1, 4, fake, fake, None, 0, None) == E_UNSUPPORTED
    # knn(xyz, n_total, new_xyz, m, offset, new_offset, b, nsample, idx, dist2, ws, ws_bytes, stream)
    for ns in (0, 101):
        assert L.pdae_seg_knn_f32(fake, 10, fake, 4, fake, fake, 2, ns, fake, fake, fake, 4096, None) == E_INVALID
    assert L.pdae_seg_knn_f32(fake, 10, fake, 0, fake, fake, 2, 8, None, None, None, 0, None) == 0  # no queries
    assert L.pdae_seg_knn_f32(fake, 10, fake, 4, None, fake, 2, 8, fake, fake, fake, 4096, None) == E_INVALID
    assert L.pdae_seg_knn_f32(fake, 10, fake, 4, fake, fake, 2, 8, fake, None, fake, 4096, None) == E_INVALID
    assert L.pdae_seg_knn_f32(fake, 10, fake, 4, fake, fake, 2, 8, fake, fake, fake, 16, None) == E_WORKSPACE
