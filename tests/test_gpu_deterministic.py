"""Deterministic gradients on the GPU: the ordered reverse index equals a stable argsort, every *_det gradient equals
the ordered-fp32 oracle bit for bit, results do not depend on batch composition, repetition or concurrent load, and
the Python layer takes the *_det entry points exactly when torch.use_deterministic_algorithms(True) is set."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import cpu_det
from pointdae_b200 import _native, chamfer_dist, dgcnn_util, ops, pointnet2_utils, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@contextlib.contextmanager
def deterministic(on=True):
    old = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(old)


def _reverse(idx, t):
    L = _native.lib()
    b, s = idx.shape
    ptr = torch.full((b, t + 1), -7, dtype=torch.int32, device=DEV)
    slot = torch.full((b, max(s, 1)), -7, dtype=torch.int32, device=DEV)
    nbytes = L.pdae_reverse_index_workspace_bytes(b, s, t)
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=DEV)
    fn = L.pdae_reverse_index_i64 if idx.dtype == torch.int64 else L.pdae_reverse_index_i32
    _native.check(fn(idx.data_ptr(), b, s, t, ptr.data_ptr(), slot.data_ptr(), ws.data_ptr(), nbytes, None), "reverse_index")
    torch.cuda.synchronize()
    return ptr.cpu().numpy(), slot.cpu().numpy()


def _check_reverse(idx_np, t):
    for dt in (torch.int32, torch.int64):
        ptr, slot = _reverse(cu(idx_np).to(dt), t)
        want_ptr, want = cpu_det.reverse_index(idx_np, t)
        assert np.array_equal(ptr, want_ptr)
        for i in range(idx_np.shape[0]):
            assert np.array_equal(slot[i, :want_ptr[i, -1]], want[i])


def _buckets(lengths, t, s, seed):
    """a cloud of s sources whose first targets receive the given bucket lengths, the rest spread at random"""
    rng = np.random.default_rng(seed)
    tgt = np.concatenate([np.full(n, p, dtype=np.int64) for p, n in enumerate(lengths)])
    rest = rng.integers(len(lengths), t, s - tgt.size)
    return rng.permutation(np.concatenate([tgt, rest]))[None]


@pytest.mark.parametrize("case", ["typical", "whole_cloud", "whole_cloud_long", "thresholds", "empty_targets", "out_of_range",
                                  "tiny_clouds"])
def test_reverse_index_is_stable_argsort(case):
    rng = np.random.default_rng(3)
    if case == "typical":
        _check_reverse(rng.integers(0, 2048, (8, 2048)), 2048)
    elif case == "whole_cloud":
        _check_reverse(np.full((3, 2048), 5), 2048)
    elif case == "whole_cloud_long":
        _check_reverse(np.full((1, 20000), 11), 100)
    elif case == "thresholds":
        _check_reverse(_buckets([1, 31, 32, 33, 63, 64, 65, 8191, 8192, 8193], 40000, 60000, 4), 40000)
    elif case == "empty_targets":
        _check_reverse(rng.integers(0, 10, (4, 3000)) * 97, 2000)
    elif case == "out_of_range":
        idx = rng.integers(0, 500, (2, 4000))
        idx[1, 123] = 500
        idx[0, 7] = -1
        _check_reverse(idx, 500)
    else:
        _check_reverse(rng.integers(0, 32, (6528, 36)), 32)


def _chamfer_case(b, n, collapsed=False, seed=1):
    c = synth.clouds(b, n, seed=seed)
    p = synth.prediction(c, seed=seed)
    if collapsed:
        p[:] = p[:, :1]
    return cu(p), cu(c)


@pytest.mark.parametrize("b,n,m,collapsed", [(128, 2048, 2048, False), (128, 2048, 2048, True), (128, 1024, 1024, False),
                                              (6528, 36, 32, False), (256, 8192, 8192, False), (1, 100000, 100000, False),
                                              (1, 20000, 20000, True)])
def test_chamfer_det_matches_ordered_oracle(b, n, m, collapsed):
    if n == m:
        x1, x2 = _chamfer_case(b, n, collapsed)
    else:
        rng = np.random.default_rng(2)
        x1, x2 = cu(rng.random((b, n, 3), dtype=np.float32)), cu(rng.random((b, m, 3), dtype=np.float32))
    d1, d2, i1, i2 = ops.chamfer_forward(x1, x2)
    rng = np.random.default_rng(5)
    g1, g2 = rng.standard_normal((b, n)).astype(np.float32), rng.standard_normal((b, m)).astype(np.float32)
    with deterministic():
        gx1, gx2 = ops.chamfer_backward(x1, x2, i1, i2, cu(g1), cu(g2))
        gone = torch.full((1,), 0.75, device=DEV)
        lx1, lx2 = ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 1.0, 0.5)
        qx1, qx2 = ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 0.5, 0.5, l1=True)
    args = [t.cpu().numpy() for t in (x1, x2, i1, i2)]
    w1, w2 = cpu_det.chamfer_bwd(*args, g1, g2)
    assert np.array_equal(gx1.cpu().numpy(), w1) and np.array_equal(gx2.cpu().numpy(), w2)
    a1, a2 = cpu_det.chamfer_loss_grad_arrays(0.75, 1.0, 0.5, b, n, m)
    w1, w2 = cpu_det.chamfer_bwd(*args, a1, a2)
    assert np.array_equal(lx1.cpu().numpy(), w1) and np.array_equal(lx2.cpu().numpy(), w2)
    a1, a2 = cpu_det.chamfer_loss_grad_arrays(0.75, 0.5, 0.5, b, n, m, d1.cpu().numpy(), d2.cpu().numpy())
    w1, w2 = cpu_det.chamfer_bwd(*args, a1, a2)
    assert np.array_equal(qx1.cpu().numpy(), w1, equal_nan=True) and np.array_equal(qx2.cpu().numpy(), w2, equal_nan=True)


def test_chamfer_det_transposed_and_wide_rows():
    rng = np.random.default_rng(6)
    b, n = 4, 700
    base = cu(rng.random((b, 3, n), dtype=np.float32))
    x1 = base.transpose(1, 2)                       # dense, read in storage order as [B][N][3]
    x2 = cu(rng.random((b, n, 6), dtype=np.float32))  # width-6 rows: the first B*N*3 floats
    d1, d2, i1, i2 = ops.chamfer_forward(x1, x2)
    g1, g2 = rng.standard_normal((b, n)).astype(np.float32), rng.standard_normal((b, n)).astype(np.float32)
    with deterministic():
        gx1, gx2 = ops.chamfer_backward(x1, x2, i1, i2, cu(g1), cu(g2))
    raw1 = base.cpu().numpy().reshape(-1)[: b * n * 3].reshape(b, n, 3)
    raw2 = x2.cpu().numpy().reshape(-1)[: b * n * 3].reshape(b, n, 3)
    w1, w2 = cpu_det.chamfer_bwd(raw1, raw2, i1.cpu().numpy(), i2.cpu().numpy(), g1, g2)
    assert np.array_equal(gx1.transpose(1, 2).contiguous().cpu().numpy().reshape(-1), w1.reshape(-1))
    flat2 = gx2.cpu().numpy().reshape(-1)
    assert np.array_equal(flat2[: b * n * 3], w2.reshape(-1)) and not flat2[b * n * 3:].any()


def test_gather_group_interp_det_match_ordered_oracle():
    rng = np.random.default_rng(7)
    # gather grad at C2 (128 clouds of 1024, 64 centres), channels 3
    b, c, n, m = 128, 3, 1024, 64
    idx = cu(rng.integers(0, n, (b, m)).astype(np.int32))
    go = cu(rng.standard_normal((b, c, m)).astype(np.float32))
    with deterministic():
        got = ops.gather_points_grad(go, idx, n)
    assert np.array_equal(got.cpu().numpy(), cpu_det.gather_grad(go.cpu().numpy(), idx.cpu().numpy(), n))
    # group_points grad at the 3DETR shape: 16 x 20000, 2048 centres x 64, with ball-query style padding (repeats)
    b, c, n, p, s = 16, 3, 20000, 2048, 64
    first = rng.integers(0, n, (b, p, 1))
    gi = np.where(rng.random((b, p, s)) < 0.5, first, rng.integers(0, n, (b, p, s))).astype(np.int32)
    gg = rng.standard_normal((b, c, p, s)).astype(np.float32)
    with deterministic():
        got = ops.group_points_grad(cu(gg), cu(gi), n)
    assert np.array_equal(got.cpu().numpy(), cpu_det.group_points_grad(gg, gi, n))
    # three_interpolate grad: 16 clouds, 4096 -> 1024 points, 64 channels
    b, c, n, m = 16, 64, 4096, 1024
    ti = rng.integers(0, m, (b, n, 3)).astype(np.int32)
    tw = rng.random((b, n, 3)).astype(np.float32)
    gt = rng.standard_normal((b, c, n)).astype(np.float32)
    with deterministic():
        got = ops.three_interpolate_grad(cu(gt), cu(ti), cu(tw), m)
    assert np.array_equal(got.cpu().numpy(), cpu_det.three_interpolate_grad(gt, ti, tw, m))


@pytest.mark.parametrize("c", [64, 128, 6])
def test_graph_feature_det_matches_ordered_oracle(c):
    rng = np.random.default_rng(8)
    b, n, k = 16, 1024, 20
    x = cu(rng.standard_normal((b, c, n)).astype(np.float32))
    idx = ops.feat_knn(x, k)
    idx[0, :, 3] = 17  # a hub
    gout = cu(rng.standard_normal((b, n, k, 2 * c)).astype(np.float32))
    with deterministic():
        got = ops._graph_feature_bwd(gout, idx, c, n)
    assert np.array_equal(got.cpu().numpy(), cpu_det.graph_feature_grad(gout.cpu().numpy(), idx.cpu().numpy()))


@pytest.mark.parametrize("metric", [0, 1, 2, 3])
def test_pair_loss_det_repeatable_and_close(metric):
    x1, x2 = _chamfer_case(32, 1024)
    _, _, i1, i2 = ops.chamfer_forward(x1, x2)
    rng = np.random.default_rng(9)
    a = cu(rng.standard_normal((32, 1024, 3)).astype(np.float32)).requires_grad_(True)
    bb = cu(rng.standard_normal((32, 1024, 3)).astype(np.float32)).requires_grad_(True)

    def grads():
        loss = ops.MatchedPairLoss.apply(a, bb, i1, i2, metric)
        return torch.autograd.grad(loss, (a, bb))

    with deterministic():
        r1, r2 = grads(), grads()
    ref = grads()
    for u, v, w in zip(r1, r2, ref):
        assert torch.equal(u, v)
        assert torch.allclose(u, w, rtol=1e-6, atol=1e-6 * float(w.abs().max()))


def test_independent_of_batch_repetition_and_load():
    x1, x2 = _chamfer_case(128, 2048)
    d1, d2, i1, i2 = ops.chamfer_forward(x1, x2)
    gone = torch.ones(1, device=DEV)
    with deterministic():
        full = ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 128.0, 128.0)
        again = ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 128.0, 128.0)
        k = 37
        one = ops.chamfer_loss_backward(x1[k:k + 1].contiguous(), x2[k:k + 1].contiguous(), i1[k:k + 1].contiguous(),
                                        i2[k:k + 1].contiguous(), d1[k:k + 1].contiguous(), d2[k:k + 1].contiguous(), gone, 1.0,
                                        1.0)
    side = torch.cuda.Stream()
    big = torch.randn(8192, 8192, device=DEV)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):  # another kernel occupies the GPU (cuBLAS: outside the deterministic region)
        for _ in range(4):
            big = big @ big * 1e-4
    with deterministic():
        loaded = ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 128.0, 128.0)
    torch.cuda.synchronize()
    for u, v, w in zip(full, again, loaded):
        assert torch.equal(u, v) and torch.equal(u, w)
    assert torch.equal(one[0][0], full[0][k]) and torch.equal(one[1][0], full[1][k])


class _Recorder:
    """wraps the loaded library and records which pdae_* symbols are called"""

    def __init__(self, lib):
        self._lib, self.called = lib, set()

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name.startswith("pdae_") and callable(fn):
            def wrapped(*a, _fn=fn, _name=name):
                self.called.add(_name)
                return _fn(*a)
            return wrapped
        return fn


def _surface_grads():
    torch.manual_seed(0)
    out = []
    x1, x2 = _chamfer_case(8, 512)
    for loss in (chamfer_dist.ChamferDistanceL2(), chamfer_dist.ChamferDistanceL1()):
        p = x1.clone().requires_grad_(True)
        out.append(torch.autograd.grad(loss(p, x2), p)[0])
    p = x1.clone().requires_grad_(True)
    nr = torch.randn(8, 512, 3, device=DEV, requires_grad=True)
    ng = torch.randn(8, 512, 3, device=DEV)
    l0, l1 = chamfer_dist.ChamferDistanceL2_withnormal()(p, x2, nr, ng)
    out += list(torch.autograd.grad(l0 + l1, (p, nr)))
    feats = torch.randn(4, 16, 1024, device=DEV, requires_grad=True)
    idx = torch.randint(0, 1024, (4, 256), device=DEV, dtype=torch.int32)
    out.append(torch.autograd.grad(pointnet2_utils.gather_operation(feats, idx).square().sum(), feats)[0])
    gidx = torch.randint(0, 64, (4, 256, 32), device=DEV, dtype=torch.int32)
    out.append(torch.autograd.grad(pointnet2_utils.grouping_operation(feats, gidx).square().sum(), feats)[0])
    tidx = torch.randint(0, 1024, (4, 2048, 3), device=DEV, dtype=torch.int32)
    tw = torch.rand(4, 2048, 3, device=DEV)
    out.append(torch.autograd.grad(pointnet2_utils.three_interpolate(feats, tidx, tw).square().sum(), feats)[0])
    x = torch.randn(4, 64, 512, device=DEV, requires_grad=True)
    out.append(torch.autograd.grad(dgcnn_util.get_graph_feature(x, k=20).square().sum(), x)[0])
    block = torch.nn.Sequential(torch.nn.Conv2d(128, 64, 1, bias=False), torch.nn.BatchNorm2d(64),
                                torch.nn.LeakyReLU(0.2)).to(DEV).train()
    y = dgcnn_util.edge_conv(x, block, k=20)
    out += list(torch.autograd.grad(y.square().sum(), (x, block[0].weight, block[1].weight)))
    return out


def test_python_surface_honours_the_flag(monkeypatch):
    rec = _Recorder(_native.lib())
    monkeypatch.setattr(_native, "lib", lambda: rec)
    with deterministic():
        first = _surface_grads()
        second = _surface_grads()
    det_called = set(rec.called)
    for u, v in zip(first, second):
        assert torch.equal(u, v)
    rec.called.clear()
    _surface_grads()
    off_called = set(rec.called)
    dets = {"pdae_chamfer_bwd_det_f32", "pdae_chamfer_loss_bwd_det_f32", "pdae_pair_loss_bwd_det_f32",
            "pdae_gather_grad_det_f32", "pdae_group_points_grad_det_f32", "pdae_three_interpolate_grad_det_f32",
            "pdae_graph_feature_grad_det_f32"}
    atomics = {d.replace("_det", "") for d in dets}
    assert dets <= det_called and not (atomics & det_called)
    assert atomics <= off_called and not (dets & off_called)
    assert any(n.startswith("pdae_edge_") for n in off_called) and not any(n.startswith("pdae_edge_") for n in det_called)


def test_hot_step_deterministic_equals_separate_det_calls():
    b, n, g, m = 128, 2048, 128, 32
    c = cu(synth.clouds(b, n, seed=4))
    p = cu(synth.prediction(c.cpu().numpy(), seed=4))
    gone = torch.ones(1, device=DEV)
    base = ops.hot_step(c, p, g, m, gone, buffers=ops.StepBuffers(b, n, g, m, torch.device(DEV)))
    base = {k: getattr(base, k).clone() for k in ("fps_idx", "center", "neighborhood", "dist1", "dist2", "idx1", "idx2", "loss3")}
    with deterministic():
        o = ops.hot_step(c, p, g, m, gone)
        torch.cuda.synchronize()
        gp, gc = ops.chamfer_loss_backward(p, c, o.idx1, o.idx2, o.dist1, o.dist2, gone, 1.0, 1.0)
    for k, v in base.items():
        assert torch.equal(getattr(o, k), v), k
    assert torch.equal(o.gpred, gp) and torch.equal(o.gcloud, gc)
    bufs = ops.StepBuffers(b, n, g, m, torch.device(DEV), deterministic=True)
    ops.hot_step(c, p, g, m, gone, buffers=bufs, deterministic=True)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            ops.hot_step(c, p, g, m, gone, buffers=bufs, deterministic=True)
    bufs.gpred.zero_()
    bufs.gcloud.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(bufs.gpred, gp) and torch.equal(bufs.gcloud, gc)


def test_hot_step_keeps_default_buffers_when_the_flag_turns_on():
    """buffers built with the flag off stay the caller's outputs once it is on, eagerly and inside a captured graph"""
    b, n, g, m = 64, 1024, 64, 32
    c = cu(synth.clouds(b, n, seed=6))
    p = cu(synth.prediction(c.cpu().numpy(), seed=6))
    gone = torch.ones(1, device=DEV)
    with deterministic(False):
        bufs = ops.StepBuffers(b, n, g, m, torch.device(DEV))
    assert bufs.flags == 0
    with deterministic():
        assert ops.hot_step(c, p, g, m, gone, buffers=bufs) is bufs
        torch.cuda.synchronize()
        gp, gc = ops.chamfer_loss_backward(p, c, bufs.idx1, bufs.idx2, bufs.dist1, bufs.dist2, gone, 1.0, 1.0)
        assert torch.equal(bufs.gpred, gp) and torch.equal(bufs.gcloud, gc)
        graph = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            with torch.cuda.graph(graph, stream=s):
                ops.hot_step(c, p, g, m, gone, buffers=bufs)
        bufs.gpred.zero_()
        bufs.gcloud.zero_()
        graph.replay()
        torch.cuda.synchronize()
    assert torch.equal(bufs.gpred, gp) and torch.equal(bufs.gcloud, gc)
    with deterministic():
        assert ops.StepBuffers(b, n, g, m, torch.device(DEV)).flags == 1  # the default reads the flag
