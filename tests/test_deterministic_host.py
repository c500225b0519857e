"""Deterministic gradients, host side: the ordered-fp32 oracle agrees with the fp64 oracle, the numpy reference of the
reverse index is a stable argsort, and the new entry points reject bad arguments before any CUDA call."""
import ctypes

import numpy as np
import pytest

from oracle import cpu as oracle
from oracle import cpu_det
from pointdae_b200 import _native

E_INVALID, E_WORKSPACE = -1, -3


def _close(got, want):
    scale = max(float(np.abs(want).max()), 1e-30)
    assert np.allclose(got, want, rtol=1e-5, atol=1e-5 * scale)


def test_ordered_oracle_matches_fp64_oracle():
    rng = np.random.default_rng(0)
    b, n, m = 3, 300, 200
    x1 = rng.standard_normal((b, n, 3)).astype(np.float32)
    x2 = rng.standard_normal((b, m, 3)).astype(np.float32)
    i1 = rng.integers(0, m, (b, n)).astype(np.int32)
    i2 = rng.integers(0, n, (b, m)).astype(np.int32)
    i2[0, :] = 7  # one bucket holding a whole cloud
    g1 = rng.standard_normal((b, n)).astype(np.float32)
    g2 = rng.standard_normal((b, m)).astype(np.float32)
    for got, want in zip(cpu_det.chamfer_bwd(x1, x2, i1, i2, g1, g2), oracle.chamfer_bwd(x1, x2, i1, i2, g1, g2)):
        _close(got, want)
    c = 5
    go = rng.standard_normal((b, c, m)).astype(np.float32)
    _close(cpu_det.gather_grad(go, i1[:, :m] % n, n), oracle.gather_grad(go, i1[:, :m] % n, n))
    gg = rng.standard_normal((b, c, 10, 8)).astype(np.float32)
    gi = rng.integers(0, n, (b, 10, 8)).astype(np.int32)
    _close(cpu_det.group_points_grad(gg, gi, n), oracle.group_points_grad(gg, gi, n))
    ti = rng.integers(0, m, (b, n, 3)).astype(np.int32)
    tw = rng.random((b, n, 3)).astype(np.float32)
    gt = rng.standard_normal((b, c, n)).astype(np.float32)
    _close(cpu_det.three_interpolate_grad(gt, ti, tw, m), oracle.three_interpolate_grad(gt, ti, tw, m))
    k = 6
    fi = rng.integers(0, 40, (b, 40, k)).astype(np.int64)
    gf = rng.standard_normal((b, 40, k, 2 * c)).astype(np.float32)
    _close(cpu_det.graph_feature_grad(gf, fi), oracle.graph_feature_grad(gf.transpose(0, 3, 1, 2), fi))


def test_reverse_index_reference_is_a_stable_argsort():
    rng = np.random.default_rng(1)
    idx = rng.integers(-2, 12, (4, 50))
    ptr, slots = cpu_det.reverse_index(idx, 10)
    for i in range(4):
        want = [j for p in range(10) for j in range(50) if idx[i, j] == p]  # targets ascending, sources ascending
        assert slots[i].tolist() == want
        assert ptr[i, -1] == len(want)
        for p in range(10):
            assert all(idx[i, j] == p for j in slots[i][ptr[i, p]:ptr[i, p + 1]])


P = ctypes.c_void_p(256)  # never dereferenced: every call below returns before touching memory


def _calls(ws, nbytes):
    """(name, call) for every new entry point with valid sizes (b = 2) and the given workspace"""
    L = _native.lib()
    return [
        ("chamfer", lambda: L.pdae_chamfer_bwd_det_f32(P, P, P, P, P, P, 2, 8, 8, P, P, ws, nbytes, None)),
        ("chamfer_loss", lambda: L.pdae_chamfer_loss_bwd_det_f32(P, P, P, P, P, P, P, 1.0, 1.0, 2, 8, 8, 0, P, P, ws, nbytes, None)),
        ("pair", lambda: L.pdae_pair_loss_bwd_det_f32(P, P, P, P, P, 1.0, 1.0, 2, 8, 8, 3, 1, P, P, ws, nbytes, None)),
        ("gather", lambda: L.pdae_gather_grad_det_f32(P, P, 2, 4, 8, 8, P, ws, nbytes, None)),
        ("group", lambda: L.pdae_group_points_grad_det_f32(P, P, 2, 4, 8, 4, 4, P, ws, nbytes, None)),
        ("interp", lambda: L.pdae_three_interpolate_grad_det_f32(P, P, P, 2, 4, 8, 8, P, ws, nbytes, None)),
        ("graph", lambda: L.pdae_graph_feature_grad_det_f32(P, P, 2, 4, 8, 3, P, ws, nbytes, None)),
        ("rev32", lambda: L.pdae_reverse_index_i32(P, 2, 8, 8, P, P, ws, nbytes, None)),
        ("rev64", lambda: L.pdae_reverse_index_i64(P, 2, 8, 8, P, P, ws, nbytes, None)),
    ]


def test_short_or_missing_workspace_is_rejected():
    for name, call in _calls(None, 0) + _calls(P, 16):
        assert call() == E_WORKSPACE, name


def test_workspace_queries_are_positive():
    L = _native.lib()
    assert L.pdae_chamfer_bwd_det_workspace_bytes(2, 8, 8) > 0
    assert L.pdae_pair_loss_bwd_det_workspace_bytes(2, 8, 8) > 0
    assert L.pdae_gather_grad_det_workspace_bytes(2, 8, 8) > 0
    assert L.pdae_group_points_grad_det_workspace_bytes(2, 8, 4, 4) > 0
    assert L.pdae_three_interpolate_grad_det_workspace_bytes(2, 8, 8) > 0
    assert L.pdae_graph_feature_grad_det_workspace_bytes(2, 4, 8, 3) > 0
    assert L.pdae_reverse_index_workspace_bytes(2, 8, 8) > 0
    assert L.pdae_step_ex_workspace_bytes(4, 256, 8, 16, 1) > L.pdae_step_ex_workspace_bytes(4, 256, 8, 16, 0)
    assert L.pdae_step_ex_workspace_bytes(4, 256, 8, 16, 0) == L.pdae_step_workspace_bytes(4, 256, 8, 16)


def test_negative_sizes_and_null_pointers_are_rejected():
    L = _native.lib()
    big = ctypes.c_size_t(1 << 40).value
    assert L.pdae_chamfer_bwd_det_f32(P, P, P, P, P, P, -1, 8, 8, P, P, P, big, None) == E_INVALID
    assert L.pdae_chamfer_bwd_det_f32(P, P, None, P, P, P, 2, 8, 8, P, P, P, big, None) == E_INVALID
    assert L.pdae_chamfer_loss_bwd_det_f32(P, P, P, P, P, P, None, 1.0, 1.0, 2, 8, 8, 0, P, P, P, big, None) == E_INVALID
    assert L.pdae_pair_loss_bwd_det_f32(P, P, P, P, None, 1.0, 1.0, 2, 8, 8, 3, 1, P, P, P, big, None) == E_INVALID
    assert L.pdae_gather_grad_det_f32(P, P, 2, -4, 8, 8, P, P, big, None) == E_INVALID
    assert L.pdae_gather_grad_det_f32(None, P, 2, 4, 8, 8, P, P, big, None) == E_INVALID
    assert L.pdae_group_points_grad_det_f32(P, None, 2, 4, 8, 4, 4, P, P, big, None) == E_INVALID
    assert L.pdae_three_interpolate_grad_det_f32(P, P, None, 2, 4, 8, 8, P, P, big, None) == E_INVALID
    assert L.pdae_graph_feature_grad_det_f32(P, P, 2, 4, -8, 3, P, P, big, None) == E_INVALID
    assert L.pdae_graph_feature_grad_det_f32(P, P, 2, 4, 8, 3, None, P, big, None) == E_INVALID
    assert L.pdae_reverse_index_i32(P, 2, -8, 8, P, P, P, big, None) == E_INVALID
    assert L.pdae_reverse_index_i64(None, 2, 8, 8, P, P, P, big, None) == E_INVALID
    assert L.pdae_step_ex_f32(P, P, 2, 64, 4, 8, P, P, P, P, P, P, P, P, P, P, P, P, big, 2, None) == E_INVALID  # unknown flag


def test_empty_batch_is_a_no_op():
    L = _native.lib()
    assert L.pdae_chamfer_bwd_det_f32(None, None, None, None, None, None, 0, 8, 8, None, None, None, 0, None) == 0
    assert L.pdae_chamfer_loss_bwd_det_f32(None, None, None, None, None, None, None, 1.0, 1.0, 0, 8, 8, 0, None, None, None, 0,
                                           None) == 0
    assert L.pdae_pair_loss_bwd_det_f32(None, None, None, None, None, 1.0, 1.0, 0, 8, 8, 3, 1, None, None, None, 0, None) == 0
    assert L.pdae_gather_grad_det_f32(None, None, 0, 4, 8, 8, None, None, 0, None) == 0
    assert L.pdae_group_points_grad_det_f32(None, None, 0, 4, 8, 4, 4, None, None, 0, None) == 0
    assert L.pdae_three_interpolate_grad_det_f32(None, None, None, 0, 4, 8, 8, None, None, 0, None) == 0
    assert L.pdae_graph_feature_grad_det_f32(None, None, 0, 4, 8, 3, None, None, 0, None) == 0
    assert L.pdae_reverse_index_i32(None, 0, 8, 8, None, None, None, 0, None) == 0
    assert L.pdae_reverse_index_i64(None, 0, 8, 8, None, None, None, 0, None) == 0
    assert L.pdae_step_ex_f32(None, None, 0, 64, 4, 8, None, None, None, None, None, None, None, None, None, None, None, None, 0,
                              1, None) == 0
