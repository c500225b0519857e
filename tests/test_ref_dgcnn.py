"""`knn` / `get_graph_feature` of models/dgcnn_util.py:7-36 against outputs of the reference's OWN module
(tests/golden/dgcnn_ref.npz, made on CPU by tests/golden/make_golden_dgcnn_ref.py).  The graph feature for a given
`idx` is exact (one subtraction per element); kNN is pinned on neighbour sets, as the reference ranks by the expanded
form (rounding / tie order unspecified); gradients to 1e-5 (order-free sums)."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import _golden_sample
from oracle import cpu as oracle

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = np.load(os.path.join(HERE, "golden", "dgcnn_ref.npz"))
_spec = importlib.util.spec_from_file_location("make_golden_dgcnn_ref", os.path.join(HERE, "golden", "make_golden_dgcnn_ref.py"))
gen = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(gen)
NAMES = sorted(gen.CASES)


def _sets_agree(idx, ref_idx, d_next_gap, scale):
    same = (np.sort(idx, axis=-1) == np.sort(ref_idx, axis=-1)).all(axis=-1)
    assert same.mean() > 0.99
    assert (d_next_gap[~same] <= 64 * np.finfo(np.float32).eps * scale).all()


@pytest.mark.parametrize("name", NAMES)
def test_oracle_graph_feature_equals_the_reference_module(name):
    b, c, n, k, extra = gen.CASES[name]
    x, idx = GOLD[name + "/x"], GOLD[name + "/idx"]
    feat = oracle.graph_feature(x, idx)
    np.testing.assert_array_equal(*_golden_sample.expect(GOLD, name + "/feature", feat))
    gx = oracle.graph_feature_grad(gen.upstream(name, feat.shape), idx)
    scale = np.abs(GOLD[name + "/gx"]).max()
    assert np.allclose(gx, GOLD[name + "/gx"], rtol=1e-5, atol=1e-5 * scale)
    np.testing.assert_array_equal(GOLD[name + "/idx_after_call"], idx + np.arange(b).reshape(-1, 1, 1) * n)
    xs = x[:, 6:] if extra else x
    oi, od = oracle.feat_knn(np.ascontiguousarray(xs), k + 1)
    _sets_agree(oi[:, :, :k], idx, od[:, :, k] - od[:, :, k - 1], (xs.astype(np.float64) ** 2).sum(axis=1).max())


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_gpu_get_graph_feature_equals_the_reference_module(name):
    from pointdae_b200 import dgcnn_util
    b, c, n, k, extra = gen.CASES[name]
    dev = "cuda:0"
    x = torch.from_numpy(GOLD[name + "/x"]).to(dev).requires_grad_(True)
    supplied = torch.from_numpy(GOLD[name + "/idx"]).to(dev)
    feat = dgcnn_util.get_graph_feature(x, k=k, idx=supplied)
    assert tuple(feat.shape) == (b, 2 * c, n, k) and not feat.is_contiguous()  # the reference's permuted view
    np.testing.assert_array_equal(*_golden_sample.expect(GOLD, name + "/feature", feat.detach().cpu().numpy()))
    np.testing.assert_array_equal(supplied.cpu().numpy(), GOLD[name + "/idx_after_call"])  # offset in place (:27)
    feat.backward(torch.from_numpy(gen.upstream(name, tuple(feat.shape))).to(dev))
    scale = np.abs(GOLD[name + "/gx"]).max()
    assert np.allclose(x.grad.cpu().numpy(), GOLD[name + "/gx"], rtol=1e-5, atol=1e-5 * scale)
    # idx=None: own kNN (on x[:, 6:] when extra_dim), pinned on neighbour sets
    own = dgcnn_util.get_graph_feature(x.detach(), k=k, idx=None, extra_dim=extra)
    xs = x.detach()[:, 6:] if extra else x.detach()
    gi = dgcnn_util.knn(xs, k).cpu().numpy()
    oi, od = oracle.feat_knn(np.ascontiguousarray(xs.cpu().numpy()), k + 1)
    np.testing.assert_array_equal(gi, oi[:, :, :k])
    same = (np.sort(gi, axis=-1) == np.sort(GOLD[name + "/idx"], axis=-1)).all(axis=-1)
    ok = torch.from_numpy(same).to(dev)[:, None, :, None].expand_as(own)
    want = feat.detach()  # the graph feature over the reference's neighbours, pinned to its stored values above
    assert same.mean() > 0.99
    assert torch.allclose(own.sum(dim=3)[ok[..., 0]], want.sum(dim=3)[ok[..., 0]], rtol=1e-4, atol=1e-4)
