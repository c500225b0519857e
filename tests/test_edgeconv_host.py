"""The float64 EdgeConv oracle (oracle/cpu_edgeconv.py) against torch float64 autograd of the reference's sequence on
the CPU (graph feature -> Conv2d -> BatchNorm2d -> leaky_relu -> max), its two entry points against each other, and the
argument checks of the EdgeConv entry points of the C ABI.  No GPU."""
import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import cpu_edgeconv as ce
from pointdae_b200 import _native

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3


def torch_layer(x, idx, block, slope):
    b, c, n = x.shape
    k = idx.size(2)
    xt = x.transpose(2, 1)
    neigh = torch.stack([xt[bi][idx[bi]] for bi in range(b)])  # (B,N,k,C)
    xi = xt[:, :, None, :].expand(-1, -1, k, -1)
    feature = torch.cat((neigh - xi, xi), dim=3).permute(0, 3, 1, 2)
    return F.leaky_relu(block[1](block[0](feature)), slope).max(dim=-1)[0]


def make(b, c, n, co, k, seed, affine=True, track=True, momentum=0.1):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((b, c, n))
    idx = np.stack([np.stack([rng.permutation(n)[:k] for _ in range(n)]) for _ in range(b)])  # distinct neighbours
    conv = nn.Conv2d(2 * c, co, 1, bias=False).double()
    bn = nn.BatchNorm2d(co, affine=affine, track_running_stats=track, momentum=momentum).double()
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(rng.standard_normal((co, 2 * c, 1, 1)) / np.sqrt(2 * c)))
        if affine:
            bn.weight.copy_(torch.from_numpy(rng.standard_normal(co)))  # both signs: max and min selections
            bn.bias.copy_(torch.from_numpy(rng.standard_normal(co) * 0.3))
        if track:
            bn.running_mean.copy_(torch.from_numpy(rng.standard_normal(co) * 0.2))
            bn.running_var.copy_(torch.from_numpy(rng.random(co) + 0.5))
    return x, idx, nn.Sequential(conv, bn), rng


def oracle_call(x, idx, block, slope, train, g):
    conv, bn = block
    return ce.layer_x(x, idx, conv.weight.detach().numpy()[:, :, 0, 0],
                      bn.weight.detach().numpy() if bn.affine else None, bn.bias.detach().numpy() if bn.affine else None,
                      bn.running_mean.numpy().copy() if bn.track_running_stats else None,
                      bn.running_var.numpy().copy() if bn.track_running_stats else None,
                      int(bn.num_batches_tracked) if bn.track_running_stats else 0, bn.momentum, bn.eps, slope, train, g)


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("affine,track,slope", [(True, True, 0.2), (False, True, 0.0), (True, False, 1.0), (True, True, 0.5)])
def test_x_oracle_matches_torch_float64_autograd(train, affine, track, slope):
    b, c, n, co, k = 2, 5, 40, 7, 6
    x, idx, block, rng = make(b, c, n, co, k, 3, affine, track)
    block.train(train)
    g = rng.standard_normal((b, co, n))
    want = oracle_call(x, idx, block, slope, train, g)
    xt = torch.from_numpy(x).requires_grad_(True)
    out = torch_layer(xt, torch.from_numpy(idx), block, slope)
    (out * torch.from_numpy(g)).sum().backward()
    np.testing.assert_allclose(want["out"], out.detach().numpy(), rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(want["dx"], xt.grad.numpy(), rtol=1e-10, atol=1e-12)
    np.testing.assert_allclose(want["dw"], block[0].weight.grad.numpy()[:, :, 0, 0], rtol=1e-10, atol=1e-12)
    if affine:
        np.testing.assert_allclose(want["dgamma"], block[1].weight.grad.numpy(), rtol=1e-10, atol=1e-12)
        np.testing.assert_allclose(want["dbeta"], block[1].bias.grad.numpy(), rtol=1e-10, atol=1e-12)
    if train and track:
        np.testing.assert_allclose(want["running_mean"], block[1].running_mean.numpy(), rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(want["running_var"], block[1].running_var.numpy(), rtol=1e-12, atol=1e-14)
        assert want["num_batches_tracked"] == int(block[1].num_batches_tracked) == 1
    assert (want["margin"] > 1e-9).all()  # tie-free: the comparison above is exact, not up to a flipped selection


def test_x_oracle_cumulative_momentum_over_two_calls():
    b, c, n, co, k = 2, 4, 30, 6, 5
    x, idx, block, rng = make(b, c, n, co, k, 9, momentum=None)
    block.train(True)
    rm, rv, nbt = block[1].running_mean.numpy().copy(), block[1].running_var.numpy().copy(), 0
    w = block[0].weight.detach().numpy()[:, :, 0, 0]
    for call in range(2):
        xc = x + call  # a different batch each call
        r = ce.layer_x(xc, idx, w, block[1].weight.detach().numpy(), block[1].bias.detach().numpy(), rm, rv, nbt, None)
        rm, rv, nbt = r["running_mean"], r["running_var"], r["num_batches_tracked"]
        with torch.no_grad():
            torch_layer(torch.from_numpy(xc), torch.from_numpy(idx), block, 0.2)
    assert nbt == int(block[1].num_batches_tracked) == 2
    np.testing.assert_allclose(rm, block[1].running_mean.numpy(), rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(rv, block[1].running_var.numpy(), rtol=1e-12, atol=1e-14)


def test_leaky_relu_derivative_at_zero_is_the_slope():
    """gamma = beta = 0: every BatchNorm output is exactly 0, where torch's derivative is the slope (finding of the
    kernels' `bn >= 0` test, which took 1 there)"""
    b, c, n, co, k = 1, 3, 20, 4, 4
    x, idx, block, rng = make(b, c, n, co, k, 5)
    with torch.no_grad():
        block[1].weight.zero_()
        block[1].bias.zero_()
    g = rng.standard_normal((b, co, n))
    want = oracle_call(x, idx, block, 0.2, True, g)
    xt = torch.from_numpy(x).requires_grad_(True)
    (torch_layer(xt, torch.from_numpy(idx), block, 0.2) * torch.from_numpy(g)).sum().backward()
    np.testing.assert_allclose(want["dbeta"], block[1].bias.grad.numpy(), rtol=1e-12)
    np.testing.assert_allclose(want["dbeta"], 0.2 * g.sum(axis=(0, 2)), rtol=1e-12)


def dyadic(shape, rng, bits, scale_bits):
    return rng.integers(-(1 << bits), 1 << bits, size=shape).astype(np.float64) / (1 << scale_bits)


@pytest.mark.parametrize("train", [True, False])
def test_z_and_x_entry_points_agree(train):
    """x and W dyadic with few bits, so z = [W1 x | (W2 - W1) x] is exact in fp32 and both levels see the same y"""
    rng = np.random.default_rng(17)
    b, c, n, co, k, ld = 2, 3, 50, 9, 7, 20
    x = dyadic((b, c, n), rng, 10, 6)
    w = dyadic((co, 2 * c), rng, 8, 8)
    idx = rng.integers(0, n, size=(b, n, k))
    idx[0, 3, :] = 5  # all slots on one point
    gamma = dyadic(co, rng, 4, 3)
    gamma[0], gamma[1] = 0.0, -0.0
    beta = dyadic(co, rng, 4, 4)
    rm, rv = dyadic(co, rng, 4, 4), np.abs(dyadic(co, rng, 4, 4)) + 0.5
    g = rng.standard_normal((b, co, n))
    xr = ce.layer_x(x, idx, w, gamma, beta, rm, rv, 0, 0.1, 1e-5, 0.2, train, g)
    xt = x.transpose(0, 2, 1)
    z = np.zeros((b, n, ld), np.float32)
    z[..., :co] = xt @ w[:, :c].T
    z[..., co:2 * co] = xt @ (w[:, c:] - w[:, :c]).T
    assert np.array_equal(z[..., :2 * co].astype(np.float64), np.concatenate([xt @ w[:, :c].T, xt @ (w[:, c:] - w[:, :c]).T], 2))
    zr = ce.layer_z(z, idx, co, gamma, beta, 1e-5, 0.2, train, g.transpose(0, 2, 1), rm, rv)
    if train:
        np.testing.assert_allclose(zr["mean"], xr["mean"], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(zr["var"], xr["var"], rtol=1e-12)
        np.testing.assert_allclose(zr["s1"].sum(axis=(0, 1)) + k * z[..., co:2 * co].astype(np.float64).sum(axis=(0, 1)), xr["mean"] * b * n * k,
                                   rtol=1e-12, atol=1e-9)
    # z-level rounds scale / shift to fp32 like the kernels: same slots, values within fp32 rounding
    assert np.array_equal(zr["jstar"], xr["jstar"])
    np.testing.assert_allclose(zr["out"], xr["out"], rtol=1e-6, atol=1e-6)
    for name in ("dgamma", "dbeta"):
        np.testing.assert_allclose(zr[name], xr[name], rtol=1e-5, atol=1e-6 * np.abs(xr[name]).max())
    wz = np.concatenate([w[:, :c], w[:, c:] - w[:, :c]], 0)  # dx = Wz^T [dP ; dQ]
    dx = np.einsum("bnj,jc->bcn", zr["dz"][..., :2 * co], wz)
    np.testing.assert_allclose(dx, xr["dx"], rtol=1e-5, atol=1e-6 * np.abs(xr["dx"]).max())
    assert not zr["dz"][..., 2 * co:].any()


def test_z_oracle_bounds_cover_an_fp32_evaluation():
    """the bounds are error budgets of fp32 arithmetic: the kernels' own fp32 sequence of s1 and of the forward, replayed
    in numpy on shifted inputs, stays inside them"""
    rng = np.random.default_rng(4)
    b, n, k, co = 1, 64, 8, 5
    z = (rng.standard_normal((b, n, 2 * co)) + 20).astype(np.float32)
    idx = rng.integers(0, n, size=(b, n, k))
    ga = rng.standard_normal(co).astype(np.float32)
    r = ce.layer_z(z, idx, co, ga, None, 1e-5, 0.2, True, rng.standard_normal((b, n, co)).astype(np.float32))
    p, q = z[0, :, :co], z[0, :, co:]
    s1 = np.zeros((n, co), np.float32)
    for j in range(k):
        s1 += p[idx[0, :, j]]
    assert (np.abs(s1 - r["s1"][0]) <= ce.EPS32 * (k + 8) * np.abs(p[idx[0]]).sum(1)).all()
    sgn = np.where(r["scale"] >= 0, np.float32(1), np.float32(-1))
    ext = sgn * np.max(p[idx[0]] * sgn, axis=1)
    y = r["scale"] * (ext + q) + r["shift"]  # fp32 throughout
    out32 = np.where(y >= 0, y, np.float32(0.2) * y)
    err = np.abs(out32.astype(np.float64) - r["out"][0].T)
    assert (err <= r["out_bound"][0].T).all() and err.max() > 0
    assert (r["dz_bound"][..., :2 * co] > 0).all()


def test_abi_rejects_bad_arguments():
    L = _native.lib()
    fake = 256
    # stats(z, ld, idx, b, n, k, co, partial, s1, stream)
    stats = L.pdae_edge_stats_f64
    for k in (0, 256):
        assert stats(fake, 64, fake, 2, 8, k, 32, fake, None, None) == E_INVALID
    assert stats(fake, 63, fake, 2, 8, 4, 32, fake, None, None) == E_INVALID     # ld < 2 co
    assert stats(fake, 64, fake, 2, 8, 4, 0, fake, None, None) == E_INVALID      # co = 0
    assert stats(fake, 64, fake, 65536, 8, 4, 32, fake, None, None) == E_UNSUPPORTED
    assert stats(None, 64, None, 0, 8, 4, 32, None, None, None) == 0            # b = 0: nothing to do
    assert stats(None, 64, None, 2, 0, 4, 32, None, None, None) == 0            # n = 0
    assert stats(fake, 64, fake, 2, 8, 4, 32, None, None, None) == E_INVALID    # no partial
    shifted = L.pdae_edge_stats_shifted_f64  # same arguments and checks
    for k in (0, 256):
        assert shifted(fake, 64, fake, 2, 8, k, 32, fake, None, None) == E_INVALID
    assert shifted(fake, 63, fake, 2, 8, 4, 32, fake, None, None) == E_INVALID
    assert shifted(fake, 64, fake, 65536, 8, 4, 32, fake, None, None) == E_UNSUPPORTED
    assert shifted(None, 64, None, 0, 8, 4, 32, None, None, None) == 0
    assert shifted(fake, 64, fake, 2, 8, 4, 32, None, None, None) == E_INVALID
    # forward(z, ld, idx, scale, shift, slope, b, n, k, co, out, jstar, stream)
    fwd = L.pdae_edge_forward_f32
    for k in (0, 256):
        assert fwd(fake, 64, fake, fake, fake, 0.2, 2, 8, k, 32, fake, None, None) == E_INVALID
    assert fwd(fake, 63, fake, fake, fake, 0.2, 2, 8, 4, 32, fake, None, None) == E_INVALID
    assert fwd(fake, 64, fake, fake, fake, 0.2, 65536, 8, 4, 32, fake, None, None) == E_UNSUPPORTED
    assert fwd(None, 64, None, None, None, 0.2, 0, 8, 4, 32, None, None, None) == 0
    assert fwd(None, 64, None, None, None, 0.2, 2, 0, 4, 32, None, None, None) == 0
    # backward select(z, ld, idx, jstar, g, scale, shift, mean, invstd, gamma, slope, train, b, n, k, co, partial, dz, s)
    sel = L.pdae_edge_backward_select_f32
    ok = (fake,) * 7
    for k in (0, 256):
        assert sel(fake, 64, fake, *ok, 0.2, 1, 2, 8, k, 32, fake, fake, None) == E_INVALID
    assert sel(fake, 63, fake, *ok, 0.2, 1, 2, 8, 4, 32, fake, fake, None) == E_INVALID
    assert sel(fake, 64, fake, *ok, 0.2, 1, 2, 8, 4, 0, fake, fake, None) == E_INVALID
    assert sel(fake, 64, fake, *ok, 0.2, 1, 65536, 8, 4, 32, fake, fake, None) == E_UNSUPPORTED
    assert sel(None, 64, None, *(None,) * 7, 0.2, 1, 0, 8, 4, 32, None, None, None) == 0
    assert sel(fake, 64, fake, *ok, 0.2, 1, 2, 8, 4, 32, None, fake, None) == E_INVALID  # no partial
    # dense(z, ld, idx, s1, mean, invstd, ca, cb, b, n, k, co, ws, ws_ints, dz, stream)
    dense = L.pdae_edge_backward_dense_f32
    need = int(L.pdae_edge_reverse_workspace_ints(2, 8, 4))
    assert need == 2 * (2 * 8 + 1 + 8 * 4)
    assert L.pdae_edge_reverse_workspace_ints(0, 8, 4) == 0
    assert dense(fake, 64, fake, *(fake,) * 5, 2, 8, 4, 32, fake, need - 1, fake, None) == E_WORKSPACE
    assert dense(fake, 64, fake, *(fake,) * 5, 2, 8, 256, 32, fake, need, fake, None) == E_INVALID
    assert dense(fake, 63, fake, *(fake,) * 5, 2, 8, 4, 32, fake, need, fake, None) == E_INVALID
    assert dense(None, 64, None, *(None,) * 5, 2, 0, 4, 32, None, 0, None, None) == 0
    # atomic backward(z, ld, idx, jstar, g, scale, shift, mean, invstd, gamma, ca, cb, slope, train, b, n, k, co, partial, dz, s)
    bwd = L.pdae_edge_backward_f32
    assert bwd(fake, 64, fake, *(fake,) * 9, 0.2, 1, 2, 8, 4, 32, fake, fake, None) == E_INVALID  # both phases at once
    assert bwd(fake, 64, fake, *(fake,) * 9, 0.2, 1, 2, 8, 0, 32, fake, None, None) == E_INVALID
    # bn_prepare(partial, np, co, m, gamma, beta, rm, rv, momentum, eps, train, mean, invstd, scale, shift, stream)
    prep = L.pdae_edge_bn_prepare_f32
    assert prep(fake, 0, 32, 100.0, fake, fake, fake, fake, 0.1, 1e-5, 1, fake, fake, fake, fake, None) == E_INVALID
    assert prep(fake, 4, 0, 100.0, fake, fake, fake, fake, 0.1, 1e-5, 1, fake, fake, fake, fake, None) == E_INVALID
    assert prep(None, 0, 32, 100.0, fake, fake, None, None, 0.1, 1e-5, 0, fake, fake, fake, fake, None) == E_INVALID
    assert L.pdae_edge_bn_backward_f32(fake, 0, 32, 100.0, fake, fake, fake, fake, fake, None) == E_INVALID
    # bn_prepare_shifted(partial, np, co, m, z, ld, gamma, beta, rm, rv, momentum, eps, train, mean, invstd, scale, shift, s)
    prep_s = L.pdae_edge_bn_prepare_shifted_f32
    out4 = (fake,) * 4
    assert prep_s(fake, 4, 32, 100.0, None, 64, fake, fake, fake, fake, 0.1, 1e-5, 1, *out4, None) == E_INVALID  # no z
    assert prep_s(fake, 4, 32, 100.0, fake, 63, fake, fake, fake, fake, 0.1, 1e-5, 1, *out4, None) == E_INVALID  # ld < 2 co
    assert prep_s(fake, 0, 32, 100.0, fake, 64, fake, fake, fake, fake, 0.1, 1e-5, 1, *out4, None) == E_INVALID  # np = 0
    assert prep_s(None, 0, 32, 100.0, None, 0, fake, fake, None, None, 0.1, 1e-5, 0, *out4, None) == E_INVALID
