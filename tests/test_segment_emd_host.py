"""Segment EMD without a GPU: the oracle (oracle/cpu_segemd.py) against the float64 transcription of the published loop
per segment, its equality with the batched equal-size oracle on equal segments, the rules for empty sides, clamped and
non-monotone offsets, and the argument checks of the C ABI."""
import numpy as np
import pytest

from oracle import cpu_emd
from oracle import cpu_segemd as se
from pointdae_b200 import _native

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3
MATCH_ATOL = 2e-3  # tests/test_emd_host.py: of the larger point mass
COST_RTOL = 1e-5


def ball(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, 3))
    x /= np.linalg.norm(x, axis=-1, keepdims=True)
    return (x * rng.random((n, 1)) ** (1.0 / 3.0)).astype(np.float32)


def mass(n, m):
    return float(max(n // m, m // n, 1))


def test_oracle_matches_float64_transcription_per_segment():
    s1, s2 = [300, 7, 1, 120], [200, 5, 3, 360]
    x1, x2 = ball(sum(s1), 1), ball(sum(s2), 2)
    o1, o2 = np.cumsum(s1).astype(np.int32), np.cumsum(s2).astype(np.int32)
    rl, rr, mats = se.match(x1, x2, o1, o2)
    cost = se.cost(x1, x2, o1, o2, rl, rr)
    assert sorted(mats) == [0, 1, 2, 3]
    for s, (lo1, hi1, lo2, hi2) in enumerate(se.segments(o1, o2, len(x1), len(x2))):
        a, b = x1[None, lo1:hi1], x2[None, lo2:hi2]
        ref = cpu_emd.match_f64(a, b)[0]
        assert np.abs(mats[s] - ref).max() <= MATCH_ATOL * mass(hi1 - lo1, hi2 - lo2)
        assert np.allclose(cost[s], cpu_emd.cost_f64(a, b, ref[None])[0], rtol=COST_RTOL, atol=1e-30)
        # the cost from the packed ratios is the cost of the accumulated match, bit for bit
        assert cost[s] == cpu_emd.cost(a, b, mats[s][None])[0]


def test_equal_segments_equal_the_batched_oracle():
    b, n, m = 3, 150, 110
    x1, x2 = ball(b * n, 3), ball(b * m, 4)
    o1 = np.arange(1, b + 1, dtype=np.int32) * n
    o2 = np.arange(1, b + 1, dtype=np.int32) * m
    rl, rr, _ = se.match(x1, x2, o1, o2)
    brl, brr, bmt = cpu_emd.match(x1.reshape(b, n, 3), x2.reshape(b, m, 3))
    # level-major (10, b*n) viewed (10, b, n) and transposed is the equal-size (b, 10, n)
    assert np.array_equal(rl.reshape(10, b, n).transpose(1, 0, 2), brl)
    assert np.array_equal(rr.reshape(10, b, m).transpose(1, 0, 2), brr)
    assert np.array_equal(se.cost(x1, x2, o1, o2, rl, rr), cpu_emd.cost(x1.reshape(b, n, 3), x2.reshape(b, m, 3), bmt))
    gc = np.array([0.5, 1.0, 2.0], np.float32)
    g1, g2 = se.grad(gc, x1, x2, o1, o2, rl, rr)
    w1, w2 = cpu_emd.grad(gc, x1.reshape(b, n, 3), x2.reshape(b, m, 3), bmt)
    assert np.array_equal(g1, w1.reshape(-1, 3)) and np.array_equal(g2, w2.reshape(-1, 3))


def test_empty_sides_and_points_past_the_end():
    x1, x2 = ball(40, 5), ball(30, 6)
    o1 = np.array([10, 10, 25, 25, 35], np.int32)  # segment 1 and 3 of xyz1 empty; rows 35.. past the end
    o2 = np.array([0, 8, 20, 30, 30], np.int32)    # segment 0 and 4 of xyz2 empty
    rl, rr, mats = se.match(x1, x2, o1, o2)
    assert sorted(mats) == [2]  # the only segment with both sides
    assert not rl[:, :10].any() and not rl[:, 25:].any() and rl[:, 10:25].any()
    assert not rr[:, :8].any() and not rr[:, 20:].any() and rr[:, 8:20].any()
    cost = se.cost(x1, x2, o1, o2, rl, rr)
    assert cost[[0, 1, 3, 4]].tolist() == [0.0] * 4 and cost[2] > 0
    g1, g2 = se.grad(np.ones(5, np.float32), x1, x2, o1, o2, rl, rr)
    assert not g1[:10].any() and not g1[25:].any() and g1[10:25].any()
    assert not g2[:8].any() and not g2[20:].any() and g2[8:20].any()


def test_clamped_and_non_monotone_offsets():
    x1, x2 = ball(50, 7), ball(40, 8)
    # offsets past the totals are clamped, and a smaller offset after a larger one gives an empty segment
    o1 = np.array([20, 12, 99], np.int32)
    o2 = np.array([15, 30, -3], np.int32)
    assert se.segments(o1, o2, 50, 40) == [(0, 20, 0, 15), (20, 20, 15, 30), (20, 50, 30, 30)]
    rl, rr, mats = se.match(x1, x2, o1, o2)
    assert sorted(mats) == [0]
    assert not rl[:, 20:].any() and not rr[:, 15:].any()
    want_l, want_r, _ = cpu_emd.match(x1[None, :20], x2[None, :15])
    assert np.array_equal(rl[:, :20], want_l[0]) and np.array_equal(rr[:, :15], want_r[0])


def test_abi_rejects_bad_arguments():
    L = _native.lib()
    f = 256  # a fake non-null pointer: every call below must return before it is used
    # count | ranges (b int4) | units of 256 points per side (+ b) | remainL (n) | remainR or rowcost (m), 256-aligned
    assert L.pdae_seg_emd_workspace_bytes(4, 100, 100) == 256 + 256 + 256 + 256 + 512 + 512
    assert L.pdae_seg_emd_workspace_bytes(0, 10, 10) == 0
    assert L.pdae_seg_emd_workspace_bytes(2, -1, 10) == 0
    # match(xyz1, n, xyz2, m, off1, off2, b, ratio_l, ratio_r, ws, ws_bytes, stream)
    for b, n, m in ((-1, 4, 4), (2, -4, 4), (2, 4, -4)):
        assert L.pdae_seg_emd_match_f32(f, n, f, m, f, f, b, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_match_f32(None, 4, None, 4, None, None, 0, None, None, None, 0, None) == 0  # b = 0: no-op
    assert L.pdae_seg_emd_match_f32(f, 4, f, 4, None, f, 2, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_match_f32(None, 4, f, 4, f, f, 2, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_match_f32(f, 4, f, 4, f, f, 2, None, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_match_f32(f, 4, f, 4, f, f, 2, f, None, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_match_f32(f, 4, f, 4, f, f, 2, f, f, None, 0, None) == E_WORKSPACE
    assert L.pdae_seg_emd_match_f32(f, 4, f, 4, f, f, 2, f, f, f, 16, None) == E_WORKSPACE
    assert L.pdae_seg_emd_match_f32(f, 1 << 28, f, 4, f, f, 2, f, f, f, 1 << 40, None) == E_UNSUPPORTED
    # cost(xyz1, n, xyz2, m, off1, off2, b, ratio_l, ratio_r, cost, ws, ws_bytes, stream)
    assert L.pdae_seg_emd_cost_f32(f, 4, f, 4, f, f, -1, f, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_f32(None, 4, None, 4, None, None, 0, None, None, None, None, 0, None) == 0
    assert L.pdae_seg_emd_cost_f32(f, 4, f, 4, f, f, 2, f, f, None, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_f32(f, 4, f, 4, f, f, 2, None, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_f32(f, 4, f, 4, f, None, 2, f, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_f32(f, 4, f, 4, f, f, 2, f, f, f, f, 8, None) == E_WORKSPACE
    # grad(grad_cost, xyz1, n, xyz2, m, off1, off2, b, ratio_l, ratio_r, grad1, grad2, ws, ws_bytes, stream)
    assert L.pdae_seg_emd_cost_grad_f32(f, f, -4, f, 4, f, f, 2, f, f, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_grad_f32(None, None, 4, None, 4, None, None, 0, None, None, None, None, None, 0, None) == 0
    assert L.pdae_seg_emd_cost_grad_f32(None, f, 4, f, 4, f, f, 2, f, f, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_grad_f32(f, f, 4, f, 4, f, f, 2, f, f, None, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_grad_f32(f, f, 4, f, 4, f, f, 2, f, f, f, None, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_grad_f32(f, f, 4, f, 4, f, f, 2, f, None, f, f, f, 1 << 20, None) == E_INVALID
    assert L.pdae_seg_emd_cost_grad_f32(f, f, 4, f, 4, f, f, 2, f, f, f, f, None, 0, None) == E_WORKSPACE
