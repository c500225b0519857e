"""EdgeConv layer on the tensor cores (ops.edge_conv: tcgen05 product + gather kernels, csrc/conv_tc.cu, csrc/edgeconv.cu)
against the reference's own sequence -- get_graph_feature -> Conv2d(2C,Co,1,bias=False) -> BatchNorm2d -> LeakyReLU(0.2)
-> max over k (models/dgcnn_util.py:96-128) -- run in true fp32 by torch on the same GPU: forward, running statistics,
and every gradient (input, convolution weight, BatchNorm weight / bias), training and eval mode."""
import pytest
import torch
import torch.nn as nn

from pointdae_b200 import dgcnn_util, ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def reference_layer(x, idx, block):
    b, c, n = x.shape
    k = idx.size(2)
    flat = (idx + torch.arange(b, device=x.device).view(-1, 1, 1) * n).view(-1)
    xt = x.transpose(2, 1).contiguous()
    neigh = xt.view(b * n, c)[flat, :].view(b, n, k, c)
    xi = xt.view(b, n, 1, c).repeat(1, 1, k, 1)
    feature = torch.cat((neigh - xi, xi), dim=3).permute(0, 3, 1, 2).contiguous()  # models/dgcnn_util.py:29-34
    return block(feature).max(dim=-1, keepdim=False)[0]


def make_block(c, co, seed):
    torch.manual_seed(seed)
    block = nn.Sequential(nn.Conv2d(2 * c, co, kernel_size=1, bias=False), nn.BatchNorm2d(co), nn.LeakyReLU(negative_slope=0.2)).to(DEV)
    with torch.no_grad():  # non-trivial affine part and statistics, some negative scales (the max becomes a min there)
        block[1].weight.copy_(torch.randn(co) * 0.7)
        block[1].bias.copy_(torch.randn(co) * 0.3)
        block[1].running_mean.copy_(torch.randn(co) * 0.2)
        block[1].running_var.copy_(torch.rand(co) + 0.5)
    return block


@pytest.mark.parametrize("b,c,n,co,k,train", [(2, 3, 512, 64, 20, True), (2, 64, 256, 64, 20, True), (1, 64, 300, 128, 20, True),
                                             (2, 128, 256, 256, 20, True), (2, 64, 256, 128, 20, False), (1, 16, 70, 24, 5, True)])
def test_edge_conv_matches_the_reference_sequence(monkeypatch, b, c, n, co, k, train):
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    g = torch.Generator(device="cpu").manual_seed(100 * c + co)
    x0 = torch.randn(b, c, n, generator=g).to(DEV)
    upstream = torch.randn(b, co, n, generator=g).to(DEV)
    idx = dgcnn_util.knn(x0, k)
    ref_block, our_block = make_block(c, co, 7), make_block(c, co, 7)
    ref_block.train(train)
    our_block.train(train)

    xr = x0.clone().requires_grad_(True)
    want = reference_layer(xr, idx, ref_block)
    (want * upstream).sum().backward()

    xo = x0.clone().requires_grad_(True)
    got = ops.edge_conv(xo, idx, our_block[0].weight, our_block[1], slope=0.2)
    (got * upstream).sum().backward()

    scale = float(want.abs().max())
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-5 * scale), float((got - want).abs().max())
    if train:
        assert torch.allclose(our_block[1].running_mean, ref_block[1].running_mean, rtol=1e-5, atol=1e-6)
        assert torch.allclose(our_block[1].running_var, ref_block[1].running_var, rtol=1e-5, atol=1e-6)
        assert int(our_block[1].num_batches_tracked) == int(ref_block[1].num_batches_tracked) == 1

    def close(a, w, what):
        s = float(w.abs().max())
        bad = ~torch.isclose(a, w, rtol=1e-4, atol=2e-5 * s)
        # the maximum routes its gradient to ONE edge: an exact or near tie may pick another edge than cuDNN's max
        assert float(bad.float().mean()) < 2e-3, (what, float(bad.float().mean()), float((a - w).abs().max()), s)

    close(xo.grad, xr.grad, "x")
    close(our_block[0].weight.grad, ref_block[0].weight.grad, "conv weight")
    close(our_block[1].weight.grad, ref_block[1].weight.grad, "bn weight")
    close(our_block[1].bias.grad, ref_block[1].bias.grad, "bn bias")


def test_no_grad_forward_keeps_nothing_and_matches():
    x = torch.randn(2, 64, 256, device=DEV)
    idx = dgcnn_util.knn(x, 20)
    block = make_block(64, 128, 3).eval()
    with torch.no_grad():
        got = ops.edge_conv(x, idx, block[0].weight, block[1])
        old = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            want = reference_layer(x, idx, block)
        finally:
            torch.backends.cudnn.allow_tf32 = old
    assert not got.requires_grad
    assert torch.allclose(got, want, rtol=1e-5, atol=1e-5 * float(want.abs().max()))


class _Encoder(nn.Module):
    """the layer structure of the reference's dgcnn_encoder (models/dgcnn_util.py:96-133), small widths"""

    def __init__(self, channel=3, widths=(16, 16, 32, 64), out=96):
        super().__init__()
        chans = [channel] + list(widths)
        for i in range(4):
            setattr(self, "conv%d" % (i + 1), nn.Sequential(nn.Conv2d(chans[i] * 2, chans[i + 1], kernel_size=1, bias=False),
                                                            nn.BatchNorm2d(chans[i + 1]), nn.LeakyReLU(negative_slope=0.2)))
        self.conv5 = nn.Sequential(nn.Conv1d(sum(widths), out, kernel_size=1, bias=False), nn.BatchNorm1d(out),
                                   nn.LeakyReLU(negative_slope=0.2))

    def forward(self, x):  # the reference's forward, on this repo's get_graph_feature
        batch_size = x.size()[0]
        feats = []
        for block in (self.conv1, self.conv2, self.conv3, self.conv4):
            x = block(dgcnn_util.get_graph_feature(x, k=20)).max(dim=-1, keepdim=False)[0]
            feats.append(x)
        x = self.conv5(torch.cat(feats, dim=1))
        return torch.nn.functional.adaptive_max_pool1d(x, 1).view(batch_size, -1)


@pytest.mark.parametrize("train", [True, False])
def test_whole_encoder_forward_and_backward(monkeypatch, train):
    """dgcnn_util.dgcnn_encoder_forward (what patch_models() binds) against the reference's forward on the same module:
    1024-d style feature, input gradient and every parameter gradient, one training step's worth."""
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    torch.manual_seed(11)
    ref, ours = _Encoder().to(DEV), _Encoder().to(DEV)
    ours.load_state_dict(ref.state_dict())
    ref.train(train)
    ours.train(train)
    x = torch.randn(3, 3, 300, device=DEV)
    xr, xo = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    want = ref(xr)
    got = dgcnn_util.dgcnn_encoder_forward(ours, xo)
    assert torch.allclose(got, want, rtol=1e-4, atol=1e-4 * float(want.abs().max())), float((got - want).abs().max())
    upstream = torch.randn_like(want)
    (want * upstream).sum().backward()
    (got * upstream).sum().backward()

    def close(a, w, what):
        # four chained layers: a 1e-6 difference in a layer's output can flip a near-tie of the NEXT layer's feature kNN or
        # of a max, which moves a few gradient entries (the strict per-layer comparison is the test above)
        s = float(w.abs().max())
        bad = ~torch.isclose(a, w, rtol=1e-3, atol=1e-4 * s)
        assert float(bad.float().mean()) < 5e-2, (what, float(bad.float().mean()), float((a - w).abs().max()), s)
        assert float((a - w).abs().max()) < 5e-3 * s, (what, float((a - w).abs().max()), s)

    close(xo.grad, xr.grad, "input")
    for (name, pr), (_, po) in zip(ref.named_parameters(), ours.named_parameters()):
        close(po.grad, pr.grad, name)
    if train:
        for (name, br), (_, bo) in zip(ref.named_buffers(), ours.named_buffers()):
            assert torch.allclose(bo.float(), br.float(), rtol=1e-4, atol=1e-5), name


def test_both_training_backward_forms_agree():
    """gather along the reversed graph (default) against the edge-parallel atomic kernel of the first version"""
    b, c, n, co, k = 2, 64, 300, 128, 20
    x = torch.randn(b, c, n, device=DEV)
    idx = dgcnn_util.knn(x, k)
    wz = torch.randn(2 * co, c, device=DEV) / c ** 0.5
    z = ops.conv1x1(x, wz, out_point_major=True)
    stats, s1 = ops.edge_stats(z, idx, co, want_s1=True)
    mean = stats[:, 0].float()
    invstd = torch.rsqrt(stats[:, 1].float() + 1e-5)
    gamma, beta = torch.randn(co, device=DEV), torch.randn(co, device=DEV)
    scale = (gamma * invstd).contiguous()
    shift = (beta - scale * mean).contiguous()
    _, jstar = ops.edge_forward(z, idx, co, scale, shift, 0.2, want_jstar=True)
    g = torch.randn(b, n, co, device=DEV)
    new = ops.edge_backward(z, idx, co, jstar, g, scale, shift, mean, invstd, gamma, 0.2, True, s1)
    old = ops.edge_backward(z, idx, co, jstar, g, scale, shift, mean, invstd, gamma, 0.2, True, None)
    for a, w in zip(new, old):
        assert torch.allclose(a, w, rtol=1e-4, atol=1e-5 * float(w.abs().max())), float((a - w).abs().max())
