"""The EdgeConv training path (csrc/edgeconv.cu) against the float64 oracle oracle/cpu_edgeconv.py.

Kernel level: edge_stats, edge_forward and the three backward forms (two-phase with s1, the atomic form without it, eval
mode) on the same fp32 z = [P | Q] as the z-level oracle -- jstar bit-exact, every other element inside the bound of its
fp32 arithmetic, no tie allowance.  End to end: ops.edge_conv against the x-level oracle with bounds from the rounding
of P and Q (eps * (|W1| |x| + |W2 - W1| |x|)) and the statistics' tolerance of 1e-5; selections whose float64 margin
lies below that rounding are counted and their flip is part of the bound of every entry they reach.

Shapes cover the 256-channel passes (co up to 512), k from 1 to the uint8 limit 255, n at the 32-point CTA edge, and
the four production layers at 16 x 2048, k = 20.  Graphs: kNN with self, duplicate slots, all slots on one point, one hub
every point lists, points nobody lists.  Inputs shifted by T (a channel mean large against its spread) test the
statistics' summation form."""
import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import cpu_edgeconv as ce
from pointdae_b200 import dgcnn_util, ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def _fp32_library_math(monkeypatch):
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)


def make_graph(kind, b, n, k, rng, pts=None):
    if kind == "knn":  # the model's graph: nearest first, self included
        pts = rng.standard_normal((b, 3, n)).astype(np.float32) if pts is None else pts
        return dgcnn_util.knn(torch.from_numpy(np.ascontiguousarray(pts)).to(DEV), k).cpu().numpy()
    idx = rng.integers(0, n, size=(b, n, k))
    if kind == "dup" and k > 1:  # duplicate slots within a row
        idx[:, :, k // 2] = idx[:, :, 0]
        idx[:, ::3, -1] = idx[:, ::3, 0]
    elif kind == "same":  # all k slots on one point
        idx[:] = rng.integers(0, n, size=(b, n, 1))
    elif kind == "hub":  # one point every point lists
        idx[:, :, rng.integers(0, k)] = n // 2
    elif kind == "orphan":  # the upper half of the points is listed by nobody
        idx = rng.integers(0, max(1, n // 2), size=(b, n, k))
    return idx.astype(np.int64)


def gammas(co, rng):
    ga = rng.standard_normal(co).astype(np.float32)  # both signs: max and min selections
    ga[0] = 0.0
    if co > 1:
        ga[1] = -0.0
    return ga


def within(got, want, bound, what):
    err = np.abs(np.asarray(got, np.float64) - want)
    bad = err > bound
    assert not bad.any(), (what, int(bad.sum()), float(err.max()), float((err / np.maximum(bound, 1e-300)).max()))
    return float((err / np.maximum(bound, 1e-300)).max())


# ---------------------------------------------------------------------------------------------------------------- kernels
KERNEL_CASES = [  # b, n, k, co, pad, graph, T
    (2, 33, 20, 1, 0, "rand", 0.0),
    (2, 31, 3, 33, 3, "dup", 5.0),
    (1, 32, 4, 255, 0, "hub", 20.0),
    (3, 33, 5, 256, 0, "orphan", 0.0),
    (2, 64, 20, 257, 5, "knn", 100.0),
    (1, 1, 1, 320, 0, "same", 0.0),
    (2, 1, 33, 64, 0, "same", 5.0),
    (1, 300, 255, 64, 0, "rand", 20.0),
    (2, 40, 33, 512, 0, "hub", 0.0),
    (1, 31, 255, 33, 0, "dup", 0.0),
    (2, 300, 20, 256, 7, "knn", 20.0),
    (1, 97, 20, 320, 0, "same", 100.0),
]


@pytest.mark.parametrize("b,n,k,co,pad,graph,T", KERNEL_CASES)
def test_kernels_match_the_z_oracle(b, n, k, co, pad, graph, T):
    rng = np.random.default_rng(1000 * co + 10 * k + n)
    ld = 2 * co + pad
    z = (rng.standard_normal((b, n, ld)) + T).astype(np.float32)
    if co >= 3:
        z[:, :, co // 2], z[:, :, co + co // 2] = T + 0.75, -0.5  # a constant channel: variance 0
    idx = make_graph(graph, b, n, k, rng)
    zt, it = torch.from_numpy(z).to(DEV), torch.from_numpy(idx).to(DEV)

    mean, var, s1 = ce.stats_z(z, idx, co)
    stats, s1_gpu = ops.edge_stats(zt, it, co, want_s1=True)
    stats = stats.cpu().numpy()
    eps = 1e-5
    inv, inv_gpu = 1 / np.sqrt(var + eps), 1 / np.sqrt(stats[:, 1] + eps)
    # statistics: invstd within 1e-5 relative, the mean within 1e-5 of the spread, each plus the fp32 rounding of
    # q_i - c_o and of v, 4 eps (max|P| + max|Q|) -- which dominates only for a channel whose spread is far below |y|
    rnd = 4 * ce.EPS32 * (np.abs(z[..., :co]).max(axis=(0, 1)) + np.abs(z[..., co:2 * co]).max(axis=(0, 1)))
    sd = np.sqrt(var + eps)
    assert np.all(np.abs(inv_gpu - inv) <= (1e-5 + rnd / sd) * inv), float((np.abs(inv_gpu - inv) / inv).max())
    assert np.all(np.abs(stats[:, 0] - mean) <= 1e-5 * sd + rnd)
    p = z[..., :co].astype(np.float64)
    within(s1_gpu.cpu().numpy(), s1, ce.EPS32 * (k + 8) * np.stack([np.abs(p[bi][idx[bi]]).sum(1) for bi in range(b)]), "s1")

    ga = gammas(co, rng)
    be = (rng.standard_normal(co) * 0.3).astype(np.float32)
    mean32, inv32 = mean.astype(np.float32), inv.astype(np.float32)
    scale32 = (ga * inv32).astype(np.float32)
    shift32 = (be - scale32 * mean32).astype(np.float32)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    for slope in (0.2, 0.0, 1.0):
        out, jstar = ops.edge_forward(zt, it, co, dev(scale32), dev(shift32), slope, want_jstar=True)
        want, wj, bound = ce.forward_z(z, idx, co, scale32, shift32, slope)
        assert np.array_equal(jstar.cpu().numpy(), wj)
        within(out.cpu().numpy(), want, bound, "out")

    g = rng.standard_normal((b, n, co)).astype(np.float32)
    args = (dev(g), dev(scale32), dev(shift32), dev(mean32), dev(inv32), dev(ga), 0.2)
    for train, use_s1 in ((True, True), (True, False), (False, False)):
        dz, dgamma, dbeta = ops.edge_backward(zt, it, co, jstar, *args, train, s1_gpu if use_s1 else None)
        want = ce.backward_z(z, idx, co, wj, g, scale32, shift32, mean32, inv32, ga, 0.2, train)
        what = "train" if train else "eval"
        within(dz.cpu().numpy(), want["dz"], want["dz_bound"], ("dz", what, use_s1))
        within(dgamma.cpu().numpy(), want["dgamma"], want["dgamma_bound"], ("dgamma", what, use_s1))
        within(dbeta.cpu().numpy(), want["dbeta"], want["dbeta_bound"], ("dbeta", what, use_s1))


# ---------------------------------------------------------------------------------------------------------------- layer
def run_layer(x, idx, c, co, rng, bn_kind="randn", slope=0.2, train=True, calls=1, momentum=0.1, eps=1e-5):
    """ops.edge_conv with an nn.BatchNorm2d configured by bn_kind against ce.layer_x; returns the ambiguous count and
    the largest error / bound ratios"""
    b, _, n = x.shape
    w = (rng.standard_normal((co, 2 * c)) / np.sqrt(2 * c)).astype(np.float32)
    bn = nn.BatchNorm2d(co, eps=eps, momentum=momentum, affine=bn_kind != "noaffine",
                        track_running_stats=bn_kind != "notrack").to(DEV)
    with torch.no_grad():
        if bn.affine:
            if bn_kind == "zero":  # zero-initialised BatchNorm: every bn output is exactly 0
                bn.weight.zero_(), bn.bias.zero_()
            else:
                bn.weight.copy_(torch.from_numpy(gammas(co, rng)))
                bn.bias.copy_(torch.from_numpy((rng.standard_normal(co) * 0.3).astype(np.float32)))
        if bn.track_running_stats:
            bn.running_mean.copy_(torch.from_numpy((rng.standard_normal(co) * 0.2).astype(np.float32)))
            bn.running_var.copy_(torch.from_numpy((rng.random(co) + 0.5).astype(np.float32)))
    bn.train(train)
    weight = torch.from_numpy(w).to(DEV).view(co, 2 * c, 1, 1).requires_grad_(True)
    it = torch.from_numpy(idx).to(DEV)
    nbt = 0
    ratios = {}
    amb = 0
    for call in range(calls):
        xc = x + np.float32(call)  # another batch per call
        rm = bn.running_mean.cpu().numpy().copy() if bn.track_running_stats else None
        rv = bn.running_var.cpu().numpy().copy() if bn.track_running_stats else None
        g = rng.standard_normal((b, co, n)).astype(np.float32)
        want = ce.layer_x(xc, idx, w, bn.weight.detach().cpu().numpy() if bn.affine else None,
                          bn.bias.detach().cpu().numpy() if bn.affine else None, rm, rv, nbt, bn.momentum, eps, slope, train,
                          g)
        xt = torch.from_numpy(xc).to(DEV).requires_grad_(True)
        weight.grad = None
        if bn.affine:
            bn.weight.grad = bn.bias.grad = None
        out = ops.edge_conv(xt, it, weight, bn, slope)
        (out * torch.from_numpy(g).to(DEV)).sum().backward()
        amb += want["ambiguous"]
        ratios["out"] = within(out.detach().cpu().numpy(), want["out"], want["out_bound"], "out")
        if "running_mean" in want:
            nbt = want["num_batches_tracked"]
            assert int(bn.num_batches_tracked) == nbt
            sd = np.sqrt(want["var"] + eps)
            # the batch mean carries the rounding of P and Q (the product's error is not zero-mean)
            mom = 1.0 / nbt if bn.momentum is None else bn.momentum
            ratios["running_mean"] = within(bn.running_mean.cpu().numpy(), want["running_mean"],
                                            1e-5 * sd + mom * want["mean_round"] + 1e-7 * np.abs(want["running_mean"]),
                                            "running_mean")
            ratios["running_var"] = within(bn.running_var.cpu().numpy(), want["running_var"], 2e-5 * (want["running_var"] + eps),
                                           "running_var")
        ratios["dx"] = within(xt.grad.cpu().numpy(), want["dx"], want["dx_bound"], "dx")
        ratios["dw"] = within(weight.grad.view(co, 2 * c).cpu().numpy(), want["dw"], want["dw_bound"], "dW")
        if bn.affine:
            ratios["dgamma"] = within(bn.weight.grad.cpu().numpy(), want["dgamma"], want["dgamma_bound"], "dgamma")
            ratios["dbeta"] = within(bn.bias.grad.cpu().numpy(), want["dbeta"], want["dbeta_bound"], "dbeta")
    return amb, ratios


LAYER_CASES = [  # b, c, n, co, k, graph, T, bn_kind, slope, train
    (2, 3, 256, 64, 20, "knn", 0.0, "randn", 0.2, True),
    (2, 1, 33, 257, 5, "dup", 5.0, "randn", 0.2, True),
    (1, 33, 31, 320, 4, "hub", 20.0, "randn", 0.0, True),
    (2, 256, 32, 33, 3, "orphan", 0.0, "randn", 1.0, True),
    (1, 3, 64, 512, 1, "rand", 100.0, "randn", 0.2, True),
    (2, 3, 300, 255, 255, "rand", 5.0, "randn", 0.2, True),
    (2, 8, 40, 16, 20, "same", 0.0, "randn", 0.2, True),
    (2, 3, 256, 64, 20, "knn", 20.0, "zero", 0.2, True),
    (2, 3, 256, 64, 20, "knn", 0.0, "noaffine", 0.2, True),
    (2, 3, 256, 64, 20, "knn", 20.0, "notrack", 0.2, True),
    (2, 3, 256, 64, 20, "knn", 20.0, "notrack", 0.2, False),
    (2, 64, 256, 128, 20, "knn", 0.0, "randn", 0.2, False),
]


@pytest.mark.parametrize("b,c,n,co,k,graph,T,bn_kind,slope,train", LAYER_CASES)
def test_edge_conv_matches_the_x_oracle(b, c, n, co, k, graph, T, bn_kind, slope, train):
    rng = np.random.default_rng(7 * co + k + c)
    x = rng.standard_normal((b, c, n)).astype(np.float32)
    idx = make_graph(graph, b, n, k, rng, x)
    amb, _ = run_layer(x + np.float32(T), idx, c, co, rng, bn_kind, slope, train,
                       eps=1e-3 if not train else 1e-5)
    assert amb <= 1e-3 * b * n * co + 2, amb  # measured: at most 14 of 32 768 selections (T = 20)


@pytest.mark.parametrize("T", [0.0, 5.0, 20.0, 100.0])
def test_statistics_hold_for_shifted_clouds(T):
    """a unit cloud shifted by T (world coordinates), momentum 1: the running buffers are the batch statistics.  Measured
    invstd error of the unshifted sums (one B200): 1.2e-6 / 5.4e-5 / 1.0e-3 at T = 5 / 20 / 100; with the shifted sums
    6.7e-7 / 4.5e-7 / 2.4e-6"""
    rng = np.random.default_rng(int(T) + 3)
    b, n, k, c, co = 2, 1024, 20, 3, 64
    x = rng.standard_normal((b, c, n)).astype(np.float32)
    idx = make_graph("knn", b, n, k, rng, x)
    run_layer(x + np.float32(T), idx, c, co, rng, momentum=1.0)


def test_positive_mean_features():
    """a previous layer's LeakyReLU output: every channel's mean well above its spread"""
    rng = np.random.default_rng(5)
    b, n, k, c, co = 2, 512, 20, 64, 128
    x = rng.standard_normal((b, c, n)).astype(np.float32)
    x = np.where(x > 0, x, 0.2 * x) * 3 + 10
    idx = make_graph("knn", b, n, k, rng, x)
    run_layer(x.astype(np.float32), idx, c, co, rng, momentum=1.0)


def test_cumulative_momentum_over_two_calls():
    rng = np.random.default_rng(8)
    x = rng.standard_normal((2, 3, 128)).astype(np.float32)
    idx = make_graph("knn", 2, 128, 20, rng, x)
    run_layer(x, idx, 3, 64, rng, momentum=None, calls=2)


def test_zero_gamma_beta_takes_the_slope_at_zero():
    """gamma = beta = 0: dbeta = slope * sum g (torch's leaky_relu'(0)); a `bn >= 0` derivative gives 5x that at 0.2
    (measured 5.000 before the fix, max error 40; after it 4.5e-7)"""
    rng = np.random.default_rng(9)
    b, c, n, co, k = 2, 3, 256, 64, 20
    x = rng.standard_normal((b, c, n)).astype(np.float32)
    idx = make_graph("knn", b, n, k, rng, x)
    bn = nn.BatchNorm2d(co).to(DEV)
    with torch.no_grad():
        bn.weight.zero_(), bn.bias.zero_()
    w = torch.randn(co, 2 * c, 1, 1, device=DEV)
    g = torch.randn(b, co, n, device=DEV)
    (ops.edge_conv(torch.from_numpy(x).to(DEV), torch.from_numpy(idx).to(DEV), w, bn, 0.2) * g).sum().backward()
    want = 0.2 * g.double().sum(dim=(0, 2))
    assert torch.allclose(bn.bias.grad.double(), want, rtol=1e-5, atol=1e-5), float((bn.bias.grad - want).abs().max())


@pytest.mark.parametrize("layer,c,co", [(1, 3, 64), (2, 64, 64), (3, 64, 128), (4, 128, 256)])
def test_production_layers(layer, c, co):
    """the DGCNN encoder's four layers at 16 x 2048 points, k = 20, kNN on the layer's input"""
    rng = np.random.default_rng(layer)
    b, n, k = 16, 2048, 20
    x = rng.standard_normal((b, c, n)).astype(np.float32)
    if layer > 1:
        x = np.where(x > 0, x, 0.2 * x).astype(np.float32)  # a LeakyReLU output, positive mean
    idx = make_graph("knn", b, n, k, rng, x)
    amb, ratios = run_layer(x, idx, c, co, rng)
    assert amb <= 1e-4 * b * n * co, amb
