"""three_nn / three_interpolate (+grad): oracle vs golden vectors of the reference's own CUDA ops (CPU), new
kernels vs golden / oracle / the live rebuilt reference (GPU).  Indices and distances bit-exact, interpolation
bit-exact (single fma chain), gradients within 1e-5 (atomics are order-free in the reference too)."""
import os

import numpy as np
import pytest
import torch

import _golden_sample
import _interp_cases
import _refmods
from oracle import cpu as oracle
from pointdae_b200 import ops, pointnet2_utils, synth

GOLD_PATH = os.path.join(os.path.dirname(__file__), "golden", "interp.npz")
CASES = _interp_cases.nn_cases(synth)


def _gold():
    return np.load(GOLD_PATH)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_cuda(name):
    z = _gold()
    unknown, known = CASES[name]
    d2, idx = oracle.three_nn(unknown, known)
    np.testing.assert_array_equal(idx, z[name + "/idx"])
    np.testing.assert_array_equal(d2, z[name + "/dist2"])
    for c in (5, 16):
        feats, weight, gout = _interp_cases.interp_inputs(synth, name, unknown, known, z[name + "/idx"], z[name + "/dist2"], c)
        np.testing.assert_array_equal(*_golden_sample.expect(z, "%s/c%d/out" % (name, c), oracle.three_interpolate(feats, idx, weight)))
        got, want = _golden_sample.expect(z, "%s/c%d/gfeats" % (name, c),
                                          oracle.three_interpolate_grad(gout, idx, weight, known.shape[1]))
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5 * np.abs(want).max())


def test_oracle_three_nn_is_a_stable_sort():
    unknown, known = CASES["ties_333_200"]
    d2, idx = oracle.three_nn(unknown, known)
    full = ((unknown[:, :, None, :].astype(np.float64) - known[:, None, :, :]) ** 2).sum(-1)
    order = np.argsort(full, axis=-1, kind="stable")[:, :, :3]
    # duplicates in `known` give exact ties: the lower index must come first
    assert (np.diff(d2, axis=-1) >= 0).all()
    tie = d2[:, :, 1:] == d2[:, :, :-1]
    assert tie.any() and (idx[:, :, 1:][tie] > idx[:, :, :-1][tie]).all()
    assert (np.sort(order, -1) == np.sort(idx, -1)).mean() > 0.99


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_gpu_three_nn_interpolate_match_golden_and_oracle(name):
    dev = torch.device("cuda:0")
    z = _gold()
    unknown, known = CASES[name]
    u, k = torch.from_numpy(unknown).to(dev), torch.from_numpy(known).to(dev)
    dist2, idx = ops.three_nn(u, k)
    np.testing.assert_array_equal(idx.cpu().numpy(), z[name + "/idx"])
    np.testing.assert_array_equal(dist2.cpu().numpy(), z[name + "/dist2"])
    dist, idx_b = pointnet2_utils.three_nn(u, k)  # public name: Euclidean distances
    np.testing.assert_array_equal(dist.cpu().numpy(), np.sqrt(z[name + "/dist2"]))
    for c in (5, 16):
        feats, weight, gout = _interp_cases.interp_inputs(synth, name, unknown, known, z[name + "/idx"], z[name + "/dist2"], c)
        f = torch.from_numpy(feats).to(dev).requires_grad_(True)
        w, g = torch.from_numpy(weight).to(dev), torch.from_numpy(gout).to(dev)
        out = pointnet2_utils.three_interpolate(f, idx, w)
        np.testing.assert_array_equal(*_golden_sample.expect(z, "%s/c%d/out" % (name, c), out.detach().cpu().numpy()))
        out.backward(g)
        got, want = _golden_sample.expect(z, "%s/c%d/gfeats" % (name, c), f.grad.cpu().numpy())
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-5 * np.abs(want).max())


@pytest.mark.gpu
def test_gpu_three_nn_large_against_live_reference_or_oracle():
    """FP-module scale (unknown 8192, known 2048, B=8): live rebuilt reference when present, oracle otherwise."""
    dev = torch.device("cuda:0")
    unknown, known = synth.clouds(8, 8192, seed=81), synth.clouds(8, 2048, seed=82)
    u, k = torch.from_numpy(unknown).to(dev), torch.from_numpy(known).to(dev)
    dist2, idx = ops.three_nn(u, k)
    ext = _refmods.ref_pointnet2()
    if ext is not None:
        rd, ri = ext.three_nn(u, k)
        assert torch.equal(idx, ri) and torch.equal(dist2, rd)
    od, oi = oracle.three_nn(unknown[:2], known[:2])
    np.testing.assert_array_equal(idx[:2].cpu().numpy(), oi)
    np.testing.assert_array_equal(dist2[:2].cpu().numpy(), od)
    # property at full size: ascending, and the first neighbour is never farther than a brute-force torch min
    assert (dist2[:, :, 1:] >= dist2[:, :, :-1]).all()
    brute = torch.cdist(u, k).min(dim=2).values
    assert torch.allclose(dist2[:, :, 0].sqrt(), brute, atol=1e-5)


@pytest.mark.gpu
def test_gpu_empty_and_error_behaviour():
    dev = torch.device("cuda:0")
    u = torch.zeros(2, 0, 3, device=dev)
    k = torch.zeros(2, 4, 3, device=dev)
    d, i = ops.three_nn(u, k)
    assert d.shape == (2, 0, 3) and i.shape == (2, 0, 3)
    d, i = ops.three_nn(k, u)  # no known points: +inf / index 0 like the reference's untouched initial values
    assert torch.isinf(d).all() and (i == 0).all()
    with pytest.raises(RuntimeError):
        ops.three_nn(k.cpu(), k.cpu())
    with pytest.raises(RuntimeError):
        ops.three_nn(k.transpose(1, 2)[:, :3].transpose(1, 2)[:, ::2], k)
