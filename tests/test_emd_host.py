"""Approximate EMD, host side: the fp32 oracle (oracle/pdae_oracle_emd.c) against a plain float64 transcription of the
published loop, the invariants of its match, its distance to the exact EMD, and argument rejection by the C ABI
without a GPU."""
import numpy as np
import pytest

from oracle import cpu_emd
from pointdae_b200 import _native

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3


def ball(b, n, seed):
    """seeded points uniform in the unit ball"""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((b, n, 3))
    x /= np.linalg.norm(x, axis=-1, keepdims=True)
    return (x * rng.random((b, n, 1)) ** (1.0 / 3.0)).astype(np.float32)


def masses(n, m):
    return (1.0, float(n // m)) if n >= m else (float(m // n), 1.0)


# Tolerances of the fp32 oracle against float64, measured on these inputs: the largest match element error is 6.4e-4
# (at (4,3000,2000); a fraction of a point's unit mass), from near-ties where remainR - sumr cancels and the fmaxf
# clamp decides; the cost, an integral over the whole match, agrees to 6.2e-7 relative.  Both bounds keep 3x / 15x
# headroom over what was measured.  The same bounds compare the GPU with this oracle (tests/test_gpu_emd.py).
MATCH_ATOL = 2e-3
COST_RTOL = 1e-5


@pytest.mark.parametrize("b,n,m", [(1, 1, 1), (3, 7, 5), (4, 1000, 3000), (4, 3000, 2000), (2, 256, 256)])
def test_oracle_matches_float64_transcription(b, n, m):
    x1, x2 = ball(b, n, 1), ball(b, m, 2)
    rl, rr, mt = cpu_emd.match(x1, x2)
    ref = cpu_emd.match_f64(x1, x2)
    assert np.abs(mt - ref).max() <= MATCH_ATOL * max(masses(n, m))
    c = cpu_emd.cost(x1, x2, mt)
    cr = cpu_emd.cost_f64(x1, x2, ref)
    assert np.allclose(c, cr, rtol=COST_RTOL, atol=1e-30)
    # the match rebuilt from the per-level ratios is the accumulated match, bit for bit
    assert np.array_equal(cpu_emd.rebuild(x1, x2, rl, rr), mt)


@pytest.mark.parametrize("b,n,m", [(3, 7, 5), (4, 1000, 3000), (4, 3000, 2000), (2, 256, 256)])
def test_match_invariants(b, n, m):
    x1, x2 = ball(b, n, 3), ball(b, m, 4)
    _, _, mt = cpu_emd.match(x1, x2)
    ml, mr = masses(n, m)
    assert (mt >= 0).all()
    eps = 4 * np.finfo(np.float32).eps * max(n, m)  # fp32 rounding of a row / column of n or m terms
    assert (mt.astype(np.float64).sum(1) <= ml * (1 + eps)).all()  # row k: sum over l
    assert (mt.astype(np.float64).sum(2) <= mr * (1 + eps)).all()  # column l: sum over k


def test_integer_division_masses():
    # 3000 vs 2000: multiR = 3000 // 2000 = 1, so a third of cloud 1's mass stays unmatched
    x1, x2 = ball(1, 300, 5), ball(1, 200, 6)
    _, _, mt = cpu_emd.match(x1, x2)
    assert mt.sum(2).max() <= 1.0 + 1e-4
    assert mt.sum() <= 200 * (1 + 1e-4)


def test_permutation_is_matched_exactly():
    # 64 points of a 0.2-spaced grid, jittered by at most 0.04: at least 0.1 apart, so at level -16384 every other
    # pair's exponent is below -87 and the first level settles the whole match
    rng = np.random.default_rng(7)
    g = np.stack(np.meshgrid(*([np.arange(4) * 0.2] * 3), indexing="ij"), -1).reshape(-1, 3)
    x1 = (g + rng.uniform(-0.02, 0.02, g.shape))[None].astype(np.float32)
    perm = rng.permutation(64)
    x2 = x1[:, perm]
    _, _, mt = cpu_emd.match(x1, x2)
    want = np.zeros((64, 64), np.float32)
    want[np.arange(64), perm] = 1.0  # match[l][k] = 1 where x2[l] = x1[k]
    assert np.allclose(mt[0], want, atol=1e-6)
    assert cpu_emd.cost(x1, x2, mt)[0] <= 1e-6


def test_ratio_to_exact_emd():
    # exact EMD of equal-size clouds is an assignment; the approximation is an upper-bound-like relaxation whose
    # ratio, measured with this oracle on these 8 seeded unit-ball pairs of 256 points, lies in [1.1997, 1.3030]
    linear_sum_assignment = pytest.importorskip("scipy.optimize").linear_sum_assignment
    x1, x2 = ball(8, 256, 10), ball(8, 256, 11)
    _, _, mt = cpu_emd.match(x1, x2)
    c = cpu_emd.cost(x1, x2, mt)
    for i in range(8):
        d = np.sqrt(((x1[i].astype(np.float64)[:, None] - x2[i].astype(np.float64)[None]) ** 2).sum(-1))
        r, cc = linear_sum_assignment(d)
        ratio = c[i] / d[r, cc].sum()
        assert 1.19 <= ratio <= 1.31, ratio


def test_abi_rejects_bad_arguments():
    L = _native.lib()
    # workspace: remainL (b,n) and remainR (b,m) floats, each 256-byte aligned; 0 for an empty or invalid shape
    assert L.pdae_emd_workspace_bytes(2, 100, 30) == 1024 + 256
    assert L.pdae_emd_workspace_bytes(128, 2048, 2048) == 2 * 128 * 2048 * 4
    assert L.pdae_emd_workspace_bytes(0, 100, 30) == 0
    assert L.pdae_emd_match_f32(None, None, -1, 4, 4, None, None, None, None, 0, None) == E_INVALID
    assert L.pdae_emd_match_f32(None, None, 2, 0, 4, None, None, None, None, 0, None) == E_INVALID
    assert L.pdae_emd_match_f32(None, None, 2, 4, 4, None, None, None, None, 0, None) == E_INVALID
    assert L.pdae_emd_match_f32(None, None, 0, 4, 4, None, None, None, None, 0, None) == 0  # empty batch: no-op
    assert L.pdae_emd_match_f32(None, None, 1, 65537, 4, None, None, None, None, 0, None) == E_UNSUPPORTED
    assert b"not supported" in L.pdae_strerror(E_UNSUPPORTED)
    assert L.pdae_emd_cost_f32(None, None, 2, 4, -4, None, None, None, None, None, 0, None) == E_INVALID
    assert L.pdae_emd_cost_f32(None, None, 0, 4, 4, None, None, None, None, None, 0, None) == 0
    assert L.pdae_emd_cost_grad_f32(None, None, None, 2, 4, 4, None, None, None, None, None, None) == E_INVALID
    assert L.pdae_emd_cost_grad_f32(None, None, None, 0, 4, 4, None, None, None, None, None, None) == 0
    # non-null clouds but no match and no ratios, or a workspace that is too small
    fake = 256
    assert L.pdae_emd_cost_f32(fake, fake, 1, 4, 4, None, None, None, fake, fake, 4096, None) == E_INVALID
    assert L.pdae_emd_match_f32(fake, fake, 1, 4, 4, fake, fake, None, fake, 16, None) == E_WORKSPACE
