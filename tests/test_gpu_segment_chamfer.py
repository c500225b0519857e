"""Segment Chamfer on the GPU (csrc/segchamfer.cu) against the oracle (oracle/cpu_segchamfer.py), bit for bit: ragged
batches with empty segments on either side, 1-point segments, sizes around the unit boundaries, a 100k-point segment,
b = 1 and b = 4096, grid ties, segment starts on every residue mod 4 and rows past the last offset.  Also the equal-size
forward, backward and losses on equal segments, the deterministic and atomic gradients, the losses against float64,
|S| = 0, and bit-identity across repeats, concurrent streams and CUDA-graph replay."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import cpu_segchamfer as cs
from pointdae_b200 import _native, chamfer_dist, ops, segment_chamfer

pytestmark = pytest.mark.gpu
DEV = "cuda"


@contextlib.contextmanager
def deterministic(on=True):
    old = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(old)


def packed(sizes, seed, grid=None, dup=False):
    rng = np.random.default_rng(seed)
    n = int(sum(sizes))
    x = (rng.integers(0, grid, (n, 3)).astype(np.float32) * 0.25) if grid else rng.random((n, 3)).astype(np.float32)
    if dup and n > 1:
        x[1::3] = x[0::3][: len(x[1::3])]
    return x, np.cumsum(sizes).astype(np.int32)


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def gpu_fwd(x1, o1, x2, o2):
    out = ops.segment_chamfer_forward(t(x1), t(x2), t(o1), t(o2))
    return [v.cpu().numpy() for v in out]


RAGGED1 = [0, 1, 127, 128, 129, 511, 512, 513, 2048, 5, 0, 1, 300]
RAGGED2 = [3, 0, 129, 1, 128, 513, 511, 2048, 512, 0, 7, 1, 40]
RESIDUE1 = [1, 64, 1, 64, 1, 64, 1, 64, 3, 128]  # 64-point segments start at rows = 1, 2, 3, 0 mod 4
RESIDUE2 = [2, 48, 1, 48, 2, 32, 3, 16, 1, 256]


def rng_sizes(b, lo, hi, seed):
    return np.random.default_rng(seed).integers(lo, hi + 1, b).tolist()


CASES = {
    "ragged": lambda: (packed(RAGGED1, 1), packed(RAGGED2, 2)),
    "residues": lambda: (packed(RESIDUE1, 3), packed(RESIDUE2, 4)),
    "b1": lambda: (packed([3000], 5), packed([2500], 6)),
    "one_100k_segment": lambda: (packed([100000], 7), packed([4096], 8)),
    "tiny_4096": lambda: (packed(rng_sizes(4096, 16, 64, 9), 9), packed(rng_sizes(4096, 16, 64, 10), 10)),
    "grid_ties": lambda: (packed([200, 0, 700, 33], 11, grid=5, dup=True), packed([150, 9, 640, 1], 12, grid=5, dup=True)),
    "object_style": lambda: (packed(rng_sizes(24, 512, 4096, 13), 13), packed(rng_sizes(24, 512, 4096, 14), 14)),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_forward_matches_oracle_bit_for_bit(case):
    (x1, o1), (x2, o2) = CASES[case]()
    got = gpu_fwd(x1, o1, x2, o2)
    want = cs.fwd(x1, x2, o1, o2)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_rows_past_the_last_offset_and_clamped_offsets():
    x1, o1 = packed([40, 0, 70], 15)
    x2, o2 = packed([33, 12, 50], 16)
    x1 = np.concatenate([x1, np.random.default_rng(1).random((37, 3)).astype(np.float32)])  # offset1[-1] < n_total
    bad1 = np.array([40, 20, 5000], np.int32)  # non-monotone and beyond n_total
    bad2 = np.array([-3, 45, 95], np.int32)
    for a, b in ((o1, o2), (bad1, bad2)):
        got = gpu_fwd(x1, a, x2, b)
        want = cs.fwd(x1, x2, a, b)
        for g, w in zip(got, want):
            assert np.array_equal(g, w)
    d1, _, i1, _ = gpu_fwd(x1, o1, x2, o2)
    assert np.all(i1[110:] == -1) and np.all(d1[110:] == 0)


@pytest.mark.parametrize("n,m", [(2048, 1024), (1024, 2048), (100, 60)])
def test_equal_segments_equal_the_equal_size_forward(n, m):
    b = 16
    x1, o1 = packed([n] * b, 17)
    x2, o2 = packed([m] * b, 18)
    d1, d2, i1, i2 = gpu_fwd(x1, o1, x2, o2)
    shift1 = (np.arange(b) * m).repeat(n).astype(np.int32)
    shift2 = (np.arange(b) * n).repeat(m).astype(np.int32)
    lib = _native.lib()
    for symmetric, tc in ((False, False), (False, True), (True, True)):  # two scans of the same body; tensor cores
        mode = lib.pdae_tune_chamfer_tc(-1 if tc else 0, 0.0)
        try:
            e1, e2, j1, j2 = [v.cpu().numpy().reshape(-1) for v in
                              ops.chamfer_forward(t(x1.reshape(b, n, 3)), t(x2.reshape(b, m, 3)), symmetric=symmetric)]
        finally:
            lib.pdae_tune_chamfer_tc(mode, 0.0)
        assert np.array_equal(d1, e1) and np.array_equal(d2, e2)
        assert np.array_equal(i1, j1 + shift1) and np.array_equal(i2, j2 + shift2)


def _ragged():
    return packed(RAGGED1, 21), packed(RAGGED2, 22)


def test_backward_det_matches_ordered_oracle_and_atomic_agrees():
    (x1, o1), (x2, o2) = _ragged()
    d1, d2, i1, i2 = gpu_fwd(x1, o1, x2, o2)
    rng = np.random.default_rng(3)
    gd1, gd2 = rng.standard_normal(len(x1)).astype(np.float32), rng.standard_normal(len(x2)).astype(np.float32)
    args = (t(x1), t(x2), t(i1), t(i2), t(gd1), t(gd2))
    with deterministic():
        g1, g2 = [v.cpu().numpy() for v in ops.segment_chamfer_backward(*args)]
    w1, w2 = cs.bwd(x1, x2, i1, i2, gd1, gd2, o1, o2)
    assert np.array_equal(g1, w1) and np.array_equal(g2, w2)
    assert not g1[i1 < 0].any() and not g2[i2 < 0].any()
    assert (i1 < 0).any() and (i2 < 0).any()
    a1, a2 = [v.cpu().numpy() for v in ops.segment_chamfer_backward(*args)]
    assert not a1[i1 < 0].any() and not a2[i2 < 0].any()
    for a, w in ((a1, w1), (a2, w2)):
        assert np.abs(a - w).max() <= 1e-6 * np.abs(w).max()


def test_backward_det_equals_equal_size_det_on_equal_segments():
    b, n, m = 8, 1024, 600
    x1, o1 = packed([n] * b, 23)
    x2, o2 = packed([m] * b, 24)
    x2[: m // 2] = x2[0]  # a long bucket: half a cloud picks one point
    d1, d2, i1, i2 = ops.segment_chamfer_forward(t(x1), t(x2), t(o1), t(o2))
    rng = np.random.default_rng(4)
    gd1, gd2 = t(rng.standard_normal(b * n).astype(np.float32)), t(rng.standard_normal(b * m).astype(np.float32))
    with deterministic():
        g1, g2 = ops.segment_chamfer_backward(t(x1), t(x2), i1, i2, gd1, gd2)
        j1 = (i1.view(b, n) - torch.arange(b, device=DEV, dtype=torch.int32).view(b, 1) * m).contiguous()
        j2 = (i2.view(b, m) - torch.arange(b, device=DEV, dtype=torch.int32).view(b, 1) * n).contiguous()
        e1, e2 = ops.chamfer_backward(t(x1.reshape(b, n, 3)), t(x2.reshape(b, m, 3)), j1, j2, gd1.view(b, n), gd2.view(b, m))
    assert torch.equal(g1, e1.view(-1, 3)) and torch.equal(g2, e2.view(-1, 3))


class _Recorder:
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


def test_deterministic_flag_selects_the_det_symbols(monkeypatch):
    (x1, o1), (x2, o2) = _ragged()
    rec = _Recorder(_native.lib())
    monkeypatch.setattr(_native, "lib", lambda: rec)

    def grads():
        a, b = t(x1).requires_grad_(True), t(x2).requires_grad_(True)
        d1, d2, _, _ = segment_chamfer.SegmentChamferFunction.apply(a, b, t(o1), t(o2))
        g = torch.autograd.grad(d1.square().sum() + d2.sum(), (a, b))
        loss = segment_chamfer.SegmentChamferDistanceL1()(a, b, t(o1), t(o2))
        return g + torch.autograd.grad(loss, (a, b))

    dets = {"pdae_seg_chamfer_bwd_det_f32", "pdae_seg_chamfer_loss_bwd_det_f32"}
    atomics = {d.replace("_det", "") for d in dets}
    with deterministic():
        grads()
    assert dets <= rec.called and not (atomics & rec.called)
    rec.called.clear()
    with deterministic(False):
        grads()
    assert atomics <= rec.called and not (dets & rec.called)


@pytest.mark.parametrize("l1", [False, True])
def test_losses_equal_the_equal_size_losses_on_equal_segments(l1):
    b, n, m = 16, 2048, 1024
    x1, o1 = packed([n] * b, 25)
    x2, o2 = packed([m] * b, 26)
    seg = (segment_chamfer.SegmentChamferDistanceL1 if l1 else segment_chamfer.SegmentChamferDistanceL2)()
    ref = (chamfer_dist.ChamferDistanceL1 if l1 else chamfer_dist.ChamferDistanceL2)()
    with deterministic():
        a, c = t(x1).requires_grad_(True), t(x2).requires_grad_(True)
        loss = seg(a, c, t(o1), t(o2))
        ga, gc = torch.autograd.grad(loss, (a, c))
        a3, c3 = t(x1.reshape(b, n, 3)).requires_grad_(True), t(x2.reshape(b, m, 3)).requires_grad_(True)
        want = ref(a3, c3)
        wa, wc = torch.autograd.grad(want, (a3, c3))
    assert abs(loss.item() - want.item()) <= 1e-6 * abs(want.item())
    assert torch.equal(ga, wa.view(-1, 3)) and torch.equal(gc, wc.view(-1, 3))


@pytest.mark.parametrize("l1", [False, True])
def test_ragged_losses_against_float64_oracle(l1):
    (x1, o1), (x2, o2) = _ragged()
    d1, d2, i1, i2 = ops.segment_chamfer_forward(t(x1), t(x2), t(o1), t(o2))
    state = torch.empty(4 * len(o1) + 1, dtype=torch.int32, device=DEV)
    loss3 = ops.segment_chamfer_loss(d1, d2, t(o1), t(o2), l1, state).cpu().numpy()
    loss, t1, t2, ns = cs.loss_f64(d1.cpu().numpy(), d2.cpu().numpy(), o1, o2, l1)
    np.testing.assert_allclose(loss3, [loss, t1, t2], rtol=1e-6)
    assert int(state[0]) == ns
    gl = torch.tensor([0.75], device=DEV)
    with deterministic():
        g1, g2 = ops.segment_chamfer_loss_backward(t(x1), t(x2), i1, i2, d1, d2, state, gl, l1)
    gd1, gd2 = cs.loss_grad_arrays(0.75, d1.cpu().numpy(), d2.cpu().numpy(), o1, o2, l1)
    w1, w2 = cs.bwd(x1, x2, i1.cpu().numpy(), i2.cpu().numpy(), gd1, gd2, o1, o2)
    assert np.array_equal(g1.cpu().numpy(), w1) and np.array_equal(g2.cpu().numpy(), w2)


@pytest.mark.parametrize("l1", [False, True])
def test_gradients_against_float64_composition(l1):
    s1, s2 = [7, 0, 13, 5, 1], [4, 9, 11, 0, 2]
    (x1, o1), (x2, o2) = packed(s1, 27), packed(s2, 28)
    a, c = t(x1).requires_grad_(True), t(x2).requires_grad_(True)
    mod = (segment_chamfer.SegmentChamferDistanceL1 if l1 else segment_chamfer.SegmentChamferDistanceL2)()
    loss = mod(a, c, t(o1), t(o2))
    ga, gc = torch.autograd.grad(loss, (a, c))
    _, _, i1, i2 = cs.fwd(x1, x2, o1, o2)
    a64, c64 = t(x1).double().requires_grad_(True), t(x2).double().requires_grad_(True)
    terms = []
    for lo1, hi1, lo2, hi2 in cs.segments(o1, o2, len(x1), len(x2)):
        if hi1 > lo1 and hi2 > lo2:
            e1 = (a64[lo1:hi1] - c64[t(i1[lo1:hi1]).long()]).square().sum(1)
            e2 = (c64[lo2:hi2] - a64[t(i2[lo2:hi2]).long()]).square().sum(1)
            if l1:
                e1, e2 = e1.sqrt(), e2.sqrt()
            terms.append((e1.mean() + e2.mean()) * (0.5 if l1 else 1.0))
    want = torch.stack(terms).mean()
    wa, wc = torch.autograd.grad(want, (a64, c64))
    assert abs(loss.item() - want.item()) <= 1e-6 * abs(want.item())
    torch.testing.assert_close(ga.double(), wa, rtol=1e-5, atol=1e-7)
    torch.testing.assert_close(gc.double(), wc, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("det", [False, True])
def test_no_valid_segment_gives_zero_loss_and_gradients(det):
    x1, o1 = packed([5, 0, 7], 29)
    x2, o2 = packed([0, 4, 0], 30)
    a, c = t(x1).requires_grad_(True), t(x2).requires_grad_(True)
    with deterministic(det):
        for mod in (segment_chamfer.SegmentChamferDistanceL2(), segment_chamfer.SegmentChamferDistanceL1()):
            loss = mod(a, c, t(o1), t(o2))
            ga, gc = torch.autograd.grad(loss, (a, c))
            assert loss.item() == 0.0
            assert torch.equal(ga, torch.zeros_like(ga)) and torch.equal(gc, torch.zeros_like(gc))


def test_mismatched_segment_counts_raise():
    x = t(np.zeros((4, 3), np.float32))
    with pytest.raises(RuntimeError, match="number of segments"):
        ops.segment_chamfer_forward(x, x, t(np.array([2, 4], np.int32)), t(np.array([4], np.int32)))


def test_reproducible_across_repeats_streams_and_graph_replay():
    (x1, o1), (x2, o2) = CASES["object_style"]()
    a, c, p, q = t(x1), t(x2), t(o1), t(o2)

    def run():
        d1, d2, i1, i2 = ops.segment_chamfer_forward(a, c, p, q)
        return [d1, d2, i1, i2, ops.segment_chamfer_loss(d1, d2, p, q)]

    ref = run()
    for _ in range(3):
        assert all(torch.equal(u, v) for u, v in zip(run(), ref))
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        r1 = run()
    with torch.cuda.stream(s2):
        r2 = run()
    torch.cuda.synchronize()
    assert all(torch.equal(u, v) for u, v in zip(r1, ref)) and all(torch.equal(u, v) for u, v in zip(r2, ref))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = run()
    for _ in range(2):
        for v in out:
            v.fill_(7)
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(u, v) for u, v in zip(out, ref))
