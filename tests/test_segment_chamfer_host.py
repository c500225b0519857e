"""Segment Chamfer without a GPU: the oracle (oracle/cpu_segchamfer.py) against float64 brute force per segment, the
rules for points without an opposite segment, the cloud-weighted loss and its gradient against torch float64 autograd,
and the argument checks of the C ABI."""
import numpy as np
import pytest
import torch

from oracle import cpu_segchamfer as cs
from pointdae_b200 import _native

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3


def packed(sizes, seed, grid=None):
    rng = np.random.default_rng(seed)
    n = int(sum(sizes))
    x = (rng.integers(0, grid, (n, 3)).astype(np.float32) * 0.25) if grid else rng.random((n, 3)).astype(np.float32)
    return x, np.cumsum(sizes).astype(np.int32)


def brute(q, r, q_lo, q_hi, r_lo, r_hi):
    """float64 squared distances of the fp32 points of one segment pair"""
    return ((q[q_lo:q_hi, None, :].astype(np.float64) - r[None, r_lo:r_hi, :]) ** 2).sum(-1)


@pytest.mark.parametrize("grid", [None, 6])
def test_oracle_matches_float64_brute_force(grid):
    s1, s2 = [5, 0, 17, 1, 33, 9, 0], [7, 3, 0, 1, 20, 40, 0]
    x1, o1 = packed(s1, 1, grid)
    x2, o2 = packed(s2, 2, grid)
    d1, d2, i1, i2 = cs.fwd(x1, x2, o1, o2)
    checked = 0
    for lo1, hi1, lo2, hi2 in cs.segments(o1, o2, len(x1), len(x2)):
        if hi1 == lo1 or hi2 == lo2:
            continue
        for q, r, ql, qh, rl, rh, dist, idx in ((x1, x2, lo1, hi1, lo2, hi2, d1, i1), (x2, x1, lo2, hi2, lo1, hi1, d2, i2)):
            d = brute(q, r, ql, qh, rl, rh)
            best = d.min(1)
            np.testing.assert_allclose(dist[ql:qh], best, rtol=3e-7, atol=1e-9)  # fp32 rounding of the same sum
            local = idx[ql:qh] - rl
            assert np.all((local >= 0) & (local < rh - rl))
            rows = np.arange(qh - ql)
            assert np.all(d[rows, local] <= best * (1 + 4e-7) + 1e-12)  # a minimiser up to fp32 rounding
            for row in rows:  # exact ties (grid clouds): the lowest index
                tied = np.flatnonzero(d[row] == best[row])
                if len(tied) > 1:
                    assert local[row] == tied[0]
            checked += qh - ql
    assert checked == 5 + 7 + 1 + 1 + 33 + 20 + 9 + 40


def test_empty_segments_and_rows_past_the_end():
    x1 = np.arange(30, dtype=np.float32).reshape(10, 3)
    x2 = np.arange(24, dtype=np.float32).reshape(8, 3) + 0.5
    o1 = np.array([3, 3, 6, 8], np.int32)  # rows 8, 9 lie past the last segment
    o2 = np.array([0, 2, 5, 8], np.int32)  # segment 0 of xyz2 is empty, segment 1 of xyz1 is empty
    d1, d2, i1, i2 = cs.fwd(x1, x2, o1, o2)
    assert i1[:3].tolist() == [-1] * 3 and d1[:3].tolist() == [0.0] * 3  # opposite segment empty
    assert i2[:2].tolist() == [-1] * 2 and d2[:2].tolist() == [0.0] * 2  # opposite segment empty
    assert i1[8:].tolist() == [-1, -1] and d1[8:].tolist() == [0.0, 0.0]  # past the last segment
    assert np.all((i1[3:6] >= 2) & (i1[3:6] < 5)) and np.all((i1[6:8] >= 5) & (i1[6:8] < 8))
    assert np.all((i2[2:5] >= 3) & (i2[2:5] < 6)) and np.all((i2[5:8] >= 6) & (i2[5:8] < 8))
    g1, g2 = cs.bwd(x1, x2, i1, i2, np.ones(10, np.float32), np.ones(8, np.float32), o1, o2)
    assert not g1[:3].any() and not g1[8:].any() and not g2[:2].any() and g1[3:8].any()
    loss, t1, t2, ns = cs.loss_f64(d1, d2, o1, o2)
    assert ns == 2 and loss == pytest.approx(t1 + t2)


def test_non_monotone_offsets_never_overlap():
    seg = cs.segments(np.array([10, 5, 20, 99], np.int32), np.array([4, 4, 2, 6], np.int32), 15, 6)
    assert seg == [(0, 10, 0, 4), (10, 10, 4, 4), (10, 15, 4, 4), (15, 15, 4, 6)]


def test_no_valid_segment_gives_zero_loss():
    d1, d2 = np.ones(4, np.float32), np.ones(3, np.float32)
    assert cs.loss_f64(d1, d2, np.array([4, 4], np.int32), np.array([0, 0], np.int32)) == (0.0, 0.0, 0.0, 0)


@pytest.mark.parametrize("l1", [False, True])
def test_loss_and_gradient_against_torch_float64(l1):
    s1, s2 = [6, 0, 11, 4, 9], [5, 7, 13, 0, 3]
    x1, o1 = packed(s1, 3)
    x2, o2 = packed(s2, 4)
    d1, d2, i1, i2 = cs.fwd(x1, x2, o1, o2)
    loss, t1, t2, ns = cs.loss_f64(d1, d2, o1, o2, l1)
    assert ns == 3
    a = torch.tensor(x1, dtype=torch.float64, requires_grad=True)
    b = torch.tensor(x2, dtype=torch.float64, requires_grad=True)
    total = 0.0
    for lo1, hi1, lo2, hi2 in cs.segments(o1, o2, len(x1), len(x2)):
        if hi1 > lo1 and hi2 > lo2:
            e1 = (a[lo1:hi1] - b[torch.from_numpy(i1[lo1:hi1].astype(np.int64))]).square().sum(1)
            e2 = (b[lo2:hi2] - a[torch.from_numpy(i2[lo2:hi2].astype(np.int64))]).square().sum(1)
            if l1:
                e1, e2 = e1.sqrt(), e2.sqrt()
            total = total + (e1.mean() + e2.mean()) * (0.5 if l1 else 1.0)
    total = total / ns
    total.backward()
    assert loss == pytest.approx(total.item(), rel=1e-6)
    gd1, gd2 = cs.loss_grad_arrays(1.0, d1, d2, o1, o2, l1)
    g1, g2 = cs.bwd(x1, x2, i1, i2, gd1, gd2, o1, o2)
    np.testing.assert_allclose(g1, a.grad.numpy(), rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(g2, b.grad.numpy(), rtol=1e-4, atol=1e-6)


def test_abi_rejects_bad_arguments():
    L = _native.lib()
    f = 256  # a fake non-null pointer: every call below must return before it is used
    assert L.pdae_seg_chamfer_fwd_workspace_bytes(0, 10, 10) == 0
    assert L.pdae_seg_chamfer_fwd_workspace_bytes(4, 100, 100) == 256 + 2 * 256
    assert L.pdae_seg_chamfer_bwd_det_workspace_bytes(0, 5) == 0
    assert L.pdae_seg_chamfer_loss_workspace_bytes(0) == 0
    assert L.pdae_seg_chamfer_loss_workspace_bytes(4) == 256
    # fwd(xyz1, n, xyz2, m, off1, off2, b, dist1, dist2, idx1, idx2, ws, ws_bytes, stream)
    for b, n, m in ((-1, 4, 4), (2, -4, 4), (2, 4, -4)):
        assert L.pdae_seg_chamfer_fwd_f32(f, n, f, m, f, f, b, f, f, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_fwd_f32(None, 4, None, 4, None, None, 0, None, None, None, None, None, 0, None) == 0
    assert L.pdae_seg_chamfer_fwd_f32(f, 4, f, 4, None, f, 2, f, f, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_fwd_f32(None, 4, f, 4, f, f, 2, f, f, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_fwd_f32(f, 4, f, 4, f, f, 2, f, None, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_fwd_f32(f, 4, f, 4, f, f, 2, f, f, f, None, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_fwd_f32(f, 4, f, 4, f, f, 2, f, f, f, f, None, 0, None) == E_WORKSPACE
    assert L.pdae_seg_chamfer_fwd_f32(f, 4, f, 4, f, f, 2, f, f, f, f, f, 16, None) == E_WORKSPACE
    assert L.pdae_seg_chamfer_fwd_f32(f, 1 << 30, f, 4, f, f, 2, f, f, f, f, f, 1 << 40, None) == E_UNSUPPORTED
    # bwd(xyz1, n, xyz2, m, idx1, idx2, gd1, gd2, gx1, gx2, [ws, ws_bytes,] stream)
    for det in (False, True):
        fn = L.pdae_seg_chamfer_bwd_det_f32 if det else L.pdae_seg_chamfer_bwd_f32
        tail = (f, 1 << 20, None) if det else (None,)
        assert fn(f, -1, f, 4, f, f, f, f, f, f, *tail) == E_INVALID
        assert fn(None, 4, f, 4, f, f, f, f, f, f, *tail) == E_INVALID
        assert fn(f, 4, f, 4, f, f, f, f, f, None, *tail) == E_INVALID
        assert fn(f, 4, f, 4, None, f, f, f, f, f, *tail) == E_INVALID
        assert fn(f, 4, f, 4, f, f, f, None, f, f, *tail) == E_INVALID
    assert L.pdae_seg_chamfer_bwd_det_f32(f, 4, f, 4, f, f, f, f, f, f, None, 0, None) == E_WORKSPACE
    assert L.pdae_seg_chamfer_bwd_det_f32(f, 4, f, 4, f, f, f, f, f, f, f, 8, None) == E_WORKSPACE
    # loss(dist1, n, dist2, m, off1, off2, b, l1, loss3, state, ws, ws_bytes, stream)
    assert L.pdae_seg_chamfer_loss_f32(f, 4, f, 4, f, f, -1, 0, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_loss_f32(f, -4, f, 4, f, f, 2, 0, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_loss_f32(None, 4, None, 4, None, None, 0, 0, None, None, None, 0, None) == 0
    assert L.pdae_seg_chamfer_loss_f32(f, 4, f, 4, None, f, 2, 0, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_loss_f32(f, 4, f, 4, f, f, 2, 0, None, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_loss_f32(f, 4, f, 4, f, f, 2, 0, f, None, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_loss_f32(f, 4, None, 4, f, f, 2, 0, f, f, f, 4096, None) == E_INVALID
    assert L.pdae_seg_chamfer_loss_f32(f, 4, f, 4, f, f, 2, 0, f, f, None, 0, None) == E_WORKSPACE
    assert L.pdae_seg_chamfer_loss_f32(f, 4, f, 4, f, f, 2, 0, f, f, f, 8, None) == E_WORKSPACE
    # loss_bwd(xyz1, n, xyz2, m, idx1, idx2, dist1, dist2, state, b, gloss, l1, gx1, gx2, [ws, ws_bytes,] stream)
    for det in (False, True):
        fn = L.pdae_seg_chamfer_loss_bwd_det_f32 if det else L.pdae_seg_chamfer_loss_bwd_f32
        tail = (f, 1 << 20, None) if det else (None,)
        assert fn(f, 4, f, 4, f, f, f, f, f, -1, f, 0, f, f, *tail) == E_INVALID
        assert fn(None, 4, None, 4, None, None, None, None, None, 0, None, 0, None, None, *tail) == 0
        assert fn(f, -4, f, 4, f, f, f, f, f, 2, f, 0, f, f, *tail) == E_INVALID
        assert fn(f, 4, f, 4, f, f, f, f, None, 2, f, 0, f, f, *tail) == E_INVALID
        assert fn(f, 4, f, 4, f, f, f, f, f, 2, None, 0, f, f, *tail) == E_INVALID
        assert fn(f, 4, f, 4, f, f, None, f, f, 2, f, 1, f, f, *tail) == E_INVALID  # L1 reads the distances
        assert fn(f, 4, f, 4, f, f, f, f, f, 2, f, 0, None, f, *tail) == E_INVALID
    assert L.pdae_seg_chamfer_loss_bwd_det_f32(f, 4, f, 4, f, f, f, f, f, 2, f, 0, f, f, None, 0, None) == E_WORKSPACE
