"""Segment EMD on the GPU (csrc/segemd.cu).

Every segment of a packed batch is specified as the equal-size EMD of that segment pair at b = 1, so the ratios, the
cost and both gradients are compared bit for bit with ops.emd_match / emd_cost / emd_cost_grad on the segment's
slices.  The shapes cover every cluster size the host picks (1, 2, 4 and 8 CTAs per segment).  Equal segments are
compared with the batched equal-size op, a few ragged segments and one segment beyond the equal-size cap with the fp32
oracle (tolerances of tests/test_gpu_emd.py, the gradient's widened for the rebuild from the ratios), and the degenerate cases, reproducibility and autograd are checked."""
import numpy as np
import pytest
import torch

from oracle import cpu_segemd as se
from pointdae_b200 import _native, emd, ops, segment_emd

pytestmark = pytest.mark.gpu

MATCH_ATOL = 2e-3   # tests/test_gpu_emd.py: of the larger point mass
COST_RTOL = 1e-5
# The oracle rebuilds the match from the ratios with exp2f where the kernels use ex2.approx (the segment op has no match
# output to compare bit for bit, unlike tests/test_gpu_emd.py): on the GPU's own ratios the cost then agrees within
# COST_RTOL and the gradients, which add rsqrtf against 1 / sqrtf, within GRAD_RTOL of the largest element.
GRAD_RTOL = 1e-4
DEV = "cuda"


def ball(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((n, 3))
    x /= np.linalg.norm(x, axis=-1, keepdims=True)
    return (x * rng.random((n, 1)) ** (1.0 / 3.0)).astype(np.float32)


def mass(n, m):
    return float(max(n // m, m // n, 1))


def packed(s1, s2, seed):
    """-> numpy x1 (N,3), x2 (M,3), int32 cumulative offsets"""
    return (ball(int(sum(s1)), seed), ball(int(sum(s2)), seed + 1), np.cumsum(s1).astype(np.int32),
            np.cumsum(s2).astype(np.int32))


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def seg_all(x1, x2, o1, o2, gc):
    """-> numpy ratios, cost and gradients of the segment op"""
    a1, a2, f1, f2, g = t(x1), t(x2), t(o1), t(o2), t(gc)
    rl, rr = ops.segment_emd_match(a1, a2, f1, f2)
    cost = ops.segment_emd_cost(a1, a2, f1, f2, rl, rr)
    g1, g2 = ops.segment_emd_cost_grad(g, a1, a2, f1, f2, rl, rr)
    return {k: v.cpu().numpy() for k, v in dict(rl=rl, rr=rr, cost=cost, g1=g1, g2=g2).items()}


def eq_all(a, b, g):
    """the equal-size op at b = 1 on one segment pair"""
    a1, a2 = t(a[None]), t(b[None])
    rl, rr, _ = ops.emd_match(a1, a2)
    cost = ops.emd_cost(a1, a2, ratio_l=rl, ratio_r=rr)
    g1, g2 = ops.emd_cost_grad(t(np.array([g], np.float32)), a1, a2, ratio_l=rl, ratio_r=rr)
    return {k: v.cpu().numpy()[0] for k, v in dict(rl=rl, rr=rr, cost=cost, g1=g1, g2=g2).items()}


def check_segments(x1, x2, o1, o2, r, gc, which=None):
    """every listed segment (default: all) equals the equal-size op on its slices, or is zero where a side is empty"""
    segs = se.segments(o1, o2, len(x1), len(x2))
    for s in (range(len(segs)) if which is None else which):
        lo1, hi1, lo2, hi2 = segs[s]
        if hi1 > lo1 and hi2 > lo2:
            w = eq_all(x1[lo1:hi1], x2[lo2:hi2], gc[s])
            assert np.array_equal(r["rl"][:, lo1:hi1], w["rl"]), s
            assert np.array_equal(r["rr"][:, lo2:hi2], w["rr"]), s
            assert r["cost"][s] == w["cost"], s
            assert np.array_equal(r["g1"][lo1:hi1], w["g1"]), s
            assert np.array_equal(r["g2"][lo2:hi2], w["g2"]), s
        else:
            assert r["cost"][s] == 0.0
            assert not r["rl"][:, lo1:hi1].any() and not r["rr"][:, lo2:hi2].any()
            assert not r["g1"][lo1:hi1].any() and not r["g2"][lo2:hi2].any()


def sizes(b, lo, hi, seed):
    return np.random.default_rng(seed).integers(lo, hi + 1, b).tolist()


# (sizes of xyz1, sizes of xyz2, segments checked or None for all)
CASES = {
    "object_128x512-4096": (sizes(128, 512, 4096, 1), sizes(128, 512, 4096, 2), None),
    "3000v2000_1000v3000": ([3000, 1000], [2000, 3000], None),
    "chunk_edges": ([1, 255, 256, 257, 511, 512, 513, 1, 300], [513, 1, 255, 512, 256, 511, 257, 1, 2], None),
    "cs1_4096x16-64": (sizes(4096, 16, 64, 3), sizes(4096, 16, 64, 4), list(range(0, 4096, 97)) + [4095]),
    "cs2_256x8192": (sizes(256, 8000, 8400, 5), sizes(256, 8000, 8400, 6), [0, 101, 255]),
    "cs4_128x2048": (sizes(128, 1900, 2048, 7), sizes(128, 1900, 2048, 8), [0, 63, 127]),
    "cs8_8x2048": (sizes(8, 2048, 2400, 9), sizes(8, 2048, 2400, 10), None),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_segments_equal_the_equal_size_op(case):
    s1, s2, which = CASES[case]
    x1, x2, o1, o2 = packed(s1, s2, 11)
    gc = np.random.default_rng(12).uniform(0.5, 2.0, len(s1)).astype(np.float32)
    check_segments(x1, x2, o1, o2, seg_all(x1, x2, o1, o2, gc), gc, which)


def test_equal_segments_equal_the_batched_op():
    b, n, m = 16, 1024, 768
    x1, x2, o1, o2 = packed([n] * b, [m] * b, 13)
    gc = np.linspace(0.5, 1.5, b).astype(np.float32)
    r = seg_all(x1, x2, o1, o2, gc)
    a1, a2 = t(x1.reshape(b, n, 3)), t(x2.reshape(b, m, 3))
    rl, rr, _ = ops.emd_match(a1, a2)
    cost = ops.emd_cost(a1, a2, ratio_l=rl, ratio_r=rr)
    g1, g2 = ops.emd_cost_grad(t(gc), a1, a2, ratio_l=rl, ratio_r=rr)
    # (10, b*n) viewed (10, b, n) and transposed is the equal-size (b, 10, n)
    assert np.array_equal(r["rl"].reshape(10, b, n).transpose(1, 0, 2), rl.cpu().numpy())
    assert np.array_equal(r["rr"].reshape(10, b, m).transpose(1, 0, 2), rr.cpu().numpy())
    assert np.array_equal(r["cost"], cost.cpu().numpy())
    assert np.array_equal(r["g1"], g1.cpu().numpy().reshape(-1, 3))
    assert np.array_equal(r["g2"], g2.cpu().numpy().reshape(-1, 3))


def close_grad(got, want):
    scale = max(float(np.nanmax(np.abs(want))), 1e-30)
    err = float(np.nanmax(np.abs(got - want))) / scale
    assert err <= GRAD_RTOL, err


def check_oracle(x1, x2, o1, o2, r, gc):
    rl, rr, mats = se.match(x1, x2, o1, o2)
    segs = se.segments(o1, o2, len(x1), len(x2))
    for s, mt in mats.items():
        lo1, hi1, lo2, hi2 = segs[s]
        assert np.abs(r["rr"][:, lo2:hi2] - rr[:, lo2:hi2]).max() <= MATCH_ATOL * mass(hi1 - lo1, hi2 - lo2)
    assert np.allclose(r["cost"], se.cost(x1, x2, o1, o2, rl, rr), rtol=COST_RTOL, atol=0)
    # on the GPU's own ratios: the cost and the gradients up to ex2.approx / rsqrtf against exp2f / 1 / sqrtf
    assert np.allclose(r["cost"], se.cost(x1, x2, o1, o2, r["rl"], r["rr"]), rtol=COST_RTOL, atol=0)
    og1, og2 = se.grad(gc, x1, x2, o1, o2, r["rl"], r["rr"])
    close_grad(r["g1"], og1)
    close_grad(r["g2"], og2)


def test_ragged_segments_against_the_oracle():
    s1, s2 = [300, 50, 1000, 0, 7], [200, 120, 700, 30, 5]
    x1, x2, o1, o2 = packed(s1, s2, 14)
    gc = np.array([1.0, 0.5, 2.0, 1.0, 1.5], np.float32)
    check_oracle(x1, x2, o1, o2, seg_all(x1, x2, o1, o2, gc), gc)


def test_segment_beyond_the_equal_size_cap():
    # 70 000 points exceed the equal-size op's 65 536; the segment op has no per-segment cap
    s1, s2 = [70000, 40], [300, 60]
    x1, x2, o1, o2 = packed(s1, s2, 15)
    gc = np.array([0.75, 1.25], np.float32)
    r = seg_all(x1, x2, o1, o2, gc)
    check_oracle(x1, x2, o1, o2, r, gc)
    check_segments(x1, x2, o1, o2, r, gc, [1])


def raw_all(x1, x2, o1, o2, gc, b):
    """the C ABI on outputs prefilled with NaN, so that every value written can be told from what was there"""
    L = _native.lib()
    a1, a2, f1, f2, g = t(x1), t(x2), t(o1), t(o2), t(gc)
    n, m = len(x1), len(x2)
    rl = torch.full((10, n), float("nan"), device=DEV)
    rr = torch.full((10, m), float("nan"), device=DEV)
    cost = torch.full((max(b, 1),), float("nan"), device=DEV)
    g1 = torch.full((n, 3), float("nan"), device=DEV)
    g2 = torch.full((m, 3), float("nan"), device=DEV)
    nb = max(L.pdae_seg_emd_workspace_bytes(b, n, m), 1)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    args = (a1.data_ptr(), n, a2.data_ptr(), m, f1.data_ptr(), f2.data_ptr(), b)
    assert L.pdae_seg_emd_match_f32(*args, rl.data_ptr(), rr.data_ptr(), ws.data_ptr(), nb, st) == 0
    assert L.pdae_seg_emd_cost_f32(*args, rl.data_ptr(), rr.data_ptr(), cost.data_ptr(), ws.data_ptr(), nb, st) == 0
    assert L.pdae_seg_emd_cost_grad_f32(g.data_ptr(), *args, rl.data_ptr(), rr.data_ptr(), g1.data_ptr(), g2.data_ptr(),
                                        ws.data_ptr(), nb, st) == 0
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in dict(rl=rl, rr=rr, cost=cost, g1=g1, g2=g2).items()}


def test_empty_sides_and_points_past_the_end():
    # empty xyz1 side, empty xyz2 side, both empty, then 25 / 9 points past the last offsets
    s1, s2 = [0, 100, 40, 0, 70], [50, 80, 0, 0, 60]
    x1, x2, o1, o2 = packed(s1 + [25], s2 + [9], 16)
    o1, o2 = o1[:-1], o2[:-1]
    gc = np.random.default_rng(17).uniform(0.5, 2.0, 5).astype(np.float32)
    r = raw_all(x1, x2, o1, o2, gc, 5)
    check_segments(x1, x2, o1, o2, r, gc)
    assert not r["rl"][:, 210:].any() and not r["g1"][210:].any()
    assert not r["rr"][:, 190:].any() and not r["g2"][190:].any()
    # the same through ops
    o = seg_all(x1, x2, o1, o2, gc)
    for k in o:
        assert np.array_equal(o[k], r[k]), k


def test_one_side_empty_everywhere():
    x1, x2 = ball(64, 18), np.zeros((0, 3), np.float32)
    o1, o2 = np.array([30, 64], np.int32), np.array([0, 0], np.int32)
    r = raw_all(x1, x2, o1, o2, np.ones(2, np.float32), 2)
    assert r["cost"].tolist() == [0.0, 0.0] and not r["rl"].any() and not r["g1"].any()


def test_clamped_and_non_monotone_offsets():
    x1, x2 = ball(900, 19), ball(700, 20)
    o1 = np.array([300, 100, 600, 10 ** 6, 5], np.int32)   # 100 < 300: an empty segment; 10**6 is clamped to 900
    o2 = np.array([250, 400, -7, 650, 700], np.int32)       # -7 is clamped to 0: an empty segment
    gc = np.random.default_rng(21).uniform(0.5, 2.0, 5).astype(np.float32)
    r = raw_all(x1, x2, o1, o2, gc, 5)
    check_segments(x1, x2, o1, o2, r, gc)


def test_no_segment():
    x1, x2 = ball(30, 22), ball(20, 23)
    # ABI: b = 0 returns 0 and writes nothing
    r = raw_all(x1, x2, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32), 0)
    assert all(np.isnan(v).all() for v in r.values())
    # ops: every point lies past the (absent) last segment
    a1, a2 = t(x1), t(x2)
    e = torch.zeros(0, dtype=torch.int32, device=DEV)
    rl, rr = ops.segment_emd_match(a1, a2, e, e)
    cost = ops.segment_emd_cost(a1, a2, e, e, rl, rr)
    g1, g2 = ops.segment_emd_cost_grad(torch.zeros(0, device=DEV), a1, a2, e, e, rl, rr)
    assert cost.shape == (0,) and not rl.any() and not rr.any() and not g1.any() and not g2.any()


def test_nan_stays_in_its_segment():
    s1, s2 = [300, 280, 500, 90], [280, 300, 260, 90]
    x1, x2, o1, o2 = packed(s1, s2, 24)
    gc = np.ones(4, np.float32)
    bad = x1.copy()
    bad[300 + 17, 1] = np.nan  # segment 1
    r_bad, r_ok = seg_all(bad, x2, o1, o2, gc), seg_all(x1, x2, o1, o2, gc)
    rows1 = np.r_[0:300, 580:1170]
    rows2 = np.r_[0:280, 580:930]
    assert np.array_equal(r_bad["rl"][:, rows1], r_ok["rl"][:, rows1])
    assert np.array_equal(r_bad["rr"][:, rows2], r_ok["rr"][:, rows2])
    assert np.array_equal(r_bad["g1"][rows1], r_ok["g1"][rows1]) and np.array_equal(r_bad["g2"][rows2], r_ok["g2"][rows2])
    assert np.array_equal(r_bad["cost"][[0, 2, 3]], r_ok["cost"][[0, 2, 3]]) and np.isnan(r_bad["cost"][1])


def test_reproducible_across_repeats_streams_flag_and_graph_replay():
    s1, s2 = sizes(24, 200, 1500, 25), sizes(24, 200, 1500, 26)
    x1, x2, o1, o2 = packed(s1, s2, 27)
    a1, a2, f1, f2 = t(x1), t(x2), t(o1), t(o2)
    gc = t(np.linspace(0.5, 1.5, 24).astype(np.float32))

    def step():
        rl, rr = ops.segment_emd_match(a1, a2, f1, f2)
        cost = ops.segment_emd_cost(a1, a2, f1, f2, rl, rr)
        g1, g2 = ops.segment_emd_cost_grad(gc, a1, a2, f1, f2, rl, rr)
        return rl, rr, cost, g1, g2

    ref = [v.clone() for v in step()]
    again = step()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        other = step()
    torch.cuda.current_stream().wait_stream(side)
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        det = step()
    finally:
        torch.use_deterministic_algorithms(prev)
    # capture succeeds only if no call synchronises with the host
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    graph.replay()
    torch.cuda.synchronize()
    for run in (again, other, det, out):
        for a, b_ in zip(ref, run):
            assert torch.equal(a, b_)


def test_autograd_equals_the_equal_size_function_per_segment():
    s1, s2 = [400, 1000, 0, 256], [700, 333, 50, 256]
    x1, x2, o1, o2 = packed(s1, s2, 28)
    a1, a2 = t(x1).requires_grad_(True), t(x2).requires_grad_(True)
    g = t(np.array([0.5, 2.0, 1.0, 1.5], np.float32))
    cost = segment_emd.segment_earth_mover_distance(a1, a2, t(o1), t(o2))
    cost.backward(g)
    for s, (lo1, hi1, lo2, hi2) in enumerate(se.segments(o1, o2, len(x1), len(x2))):
        if hi1 == lo1 or hi2 == lo2:
            assert cost[s].item() == 0.0 and not a2.grad[lo2:hi2].any()
            continue
        b1 = t(x1[None, lo1:hi1]).requires_grad_(True)
        b2 = t(x2[None, lo2:hi2]).requires_grad_(True)
        c = emd.earth_mover_distance(b1, b2)
        c.backward(g[s:s + 1])
        assert torch.equal(cost[s:s + 1].detach(), c.detach())
        assert torch.equal(a1.grad[lo1:hi1], b1.grad[0]) and torch.equal(a2.grad[lo2:hi2], b2.grad[0])
