"""Approximate EMD on the GPU (csrc/emd.cu) against the fp32 oracle (oracle/pdae_oracle_emd.c), bit-reproducibility
across paths, batch shapes, streams and the deterministic flag, degenerate inputs, the `emd_cuda` drop-in and CUDA-graph
capture.

The oracle uses libm exp2f and 1 / sqrtf where the kernels use ex2.approx and rsqrtf, so ratios and the match are
compared within the tolerance measured for the fp32 oracle against float64 (tests/test_emd_host.py), which bounds how
far a few ulps in the pair terms can move the algorithm.  Cost and gradient are then also compared with the oracle
evaluated on the GPU's own match: the cost is bit-exact there, the gradient differs by rsqrtf alone."""
import numpy as np
import pytest
import torch

from oracle import cpu_emd
from pointdae_b200 import emd, ops

pytestmark = pytest.mark.gpu

MATCH_ATOL = 2e-3   # of the larger point mass, as for the oracle against float64
COST_RTOL = 1e-5
GRAD_RTOL = 1e-5    # rsqrtf against 1 / sqrtf, relative to the largest gradient element
DEV = "cuda"


def ball(b, n, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((b, n, 3))
    x /= np.linalg.norm(x, axis=-1, keepdims=True)
    return (x * rng.random((b, n, 1)) ** (1.0 / 3.0)).astype(np.float32)


def mass(n, m):
    return float(max(n // m, m // n, 1))


def gpu_all(x1, x2, g=None):
    """-> dict of numpy results of the ratio path, plus the materialised match"""
    t1, t2 = torch.from_numpy(x1).to(DEV), torch.from_numpy(x2).to(DEV)
    rl, rr, mt = ops.emd_match(t1, t2, materialize=True)
    cost = ops.emd_cost(t1, t2, ratio_l=rl, ratio_r=rr)
    gc = torch.from_numpy(g).to(DEV) if g is not None else torch.ones(x1.shape[0], device=DEV)
    g1, g2 = ops.emd_cost_grad(gc, t1, t2, ratio_l=rl, ratio_r=rr)
    return {k: v.cpu().numpy() for k, v in dict(rl=rl, rr=rr, match=mt, cost=cost, g1=g1, g2=g2, gc=gc).items()}


def close_grad(got, want):
    scale = max(float(np.nanmax(np.abs(want))), 1e-30)
    err = float(np.nanmax(np.abs(got - want))) / scale if want.size else 0.0
    assert err <= GRAD_RTOL, err


def check_against_oracle(x1, x2, r, clouds):
    n, m = x1.shape[1], x2.shape[1]
    for i in clouds:
        a1, a2 = x1[i:i + 1], x2[i:i + 1]
        rl, rr, mt = cpu_emd.match(a1, a2)
        gm = r["match"][i:i + 1]
        assert np.abs(gm - mt).max() <= MATCH_ATOL * mass(n, m)
        assert np.abs(r["rr"][i:i + 1] - rr).max() <= MATCH_ATOL * mass(n, m)
        oc = cpu_emd.cost(a1, a2, mt)
        assert np.allclose(r["cost"][i:i + 1], oc, rtol=COST_RTOL, atol=0)
        # the same definitions on the GPU's own match: the cost bit for bit, the gradient up to rsqrtf
        assert np.array_equal(cpu_emd.cost(a1, a2, gm), r["cost"][i:i + 1])
        og1, og2 = cpu_emd.grad(r["gc"][i:i + 1], a1, a2, gm)
        close_grad(r["g1"][i:i + 1], og1)
        close_grad(r["g2"][i:i + 1], og2)
        # the materialised match is the oracle's rebuild from the GPU's ratios, up to ex2.approx against exp2f
        rb = cpu_emd.rebuild(a1, a2, r["rl"][i:i + 1], r["rr"][i:i + 1])
        assert np.abs(gm - rb).max() <= 1e-5 * mass(n, m)


@pytest.mark.parametrize("b,n,m,clouds", [
    (1, 1, 1, [0]), (3, 7, 5, [0, 1, 2]), (4, 1000, 3000, [0, 3]), (4, 3000, 2000, [1]), (2, 256, 256, [0, 1]),
    (16, 2048, 2048, [0, 15]), (128, 2048, 2048, [0, 77, 127]), (2, 8192, 8192, [1])])
def test_against_oracle(b, n, m, clouds):
    x1, x2 = ball(b, n, 20 + b), ball(b, m, 40 + b)
    g = np.random.default_rng(b).uniform(0.5, 2.0, b).astype(np.float32)
    check_against_oracle(x1, x2, gpu_all(x1, x2, g), clouds)


def test_paths_are_bit_identical():
    x1 = torch.from_numpy(ball(6, 1500, 1)).to(DEV)
    x2 = torch.from_numpy(ball(6, 1100, 2)).to(DEV)
    rl, rr, mt = ops.emd_match(x1, x2, materialize=True)
    gc = torch.linspace(0.5, 1.5, 6, device=DEV)
    assert torch.equal(ops.emd_cost(x1, x2, ratio_l=rl, ratio_r=rr), ops.emd_cost(x1, x2, match=mt))
    for a, b_ in zip(ops.emd_cost_grad(gc, x1, x2, ratio_l=rl, ratio_r=rr), ops.emd_cost_grad(gc, x1, x2, match=mt)):
        assert torch.equal(a, b_)


def test_cluster_shape_equals_batch_shape():
    # one cloud alone runs on a cluster of CTAs; inside a batch of 256 it gets one CTA
    x1 = torch.from_numpy(ball(256, 2048, 3)).to(DEV)
    x2 = torch.from_numpy(ball(256, 2048, 4)).to(DEV)
    rl, rr, _ = ops.emd_match(x1, x2)
    for i in (0, 131, 255):
        a_rl, a_rr, _ = ops.emd_match(x1[i:i + 1].contiguous(), x2[i:i + 1].contiguous())
        assert torch.equal(a_rl, rl[i:i + 1]) and torch.equal(a_rr, rr[i:i + 1])
    c = ops.emd_cost(x1, x2, ratio_l=rl, ratio_r=rr)
    c5 = ops.emd_cost(x1[5:6].contiguous(), x2[5:6].contiguous(), ratio_l=rl[5:6].contiguous(), ratio_r=rr[5:6].contiguous())
    assert torch.equal(c[5:6], c5)


def test_repeatable_beside_concurrent_work_and_under_deterministic_flag():
    x1 = torch.from_numpy(ball(8, 2048, 5)).to(DEV).requires_grad_(True)
    x2 = torch.from_numpy(ball(8, 2048, 6)).to(DEV).requires_grad_(True)

    def run():
        c = emd.earth_mover_distance(x1, x2)
        g1, g2 = torch.autograd.grad(c.sum(), (x1, x2))
        torch.cuda.synchronize()
        return c.detach(), g1, g2

    ref = run()
    again = run()
    side = torch.cuda.Stream()
    big = torch.randn(8192, 8192, device=DEV)
    with torch.cuda.stream(side):
        for _ in range(4):
            big = big @ big * 1e-4
    busy = run()
    torch.cuda.synchronize()
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        det = run()
    finally:
        torch.use_deterministic_algorithms(prev)
    for other in (again, busy, det):
        for a, b_ in zip(ref, other):
            assert torch.equal(a, b_)


def _degenerate_cases():
    rng = np.random.default_rng(9)
    same = np.tile(rng.standard_normal((1, 1, 3)), (2, 300, 1)).astype(np.float32)
    dup = rng.standard_normal((2, 50, 3)).astype(np.float32)
    dup = np.repeat(dup, 4, axis=1)  # every point four times
    far1 = ball(2, 200, 11)
    far2 = (ball(2, 150, 12) + np.float32(100.0)).astype(np.float32)  # every e below level 0 underflows
    return {"identical": (same, same[:, :200].copy()), "duplicates": (dup, ball(2, 160, 13)),
            "far_apart": (far1, far2)}


@pytest.mark.parametrize("case", ["identical", "duplicates", "far_apart"])
def test_degenerate_inputs_match_oracle(case):
    x1, x2 = _degenerate_cases()[case]
    check_against_oracle(x1, x2, gpu_all(x1, x2), range(x1.shape[0]))


def test_nan_stays_in_its_cloud():
    x1, x2 = ball(4, 300, 14), ball(4, 280, 15)
    bad = x1.copy()
    bad[2, 17, 1] = np.nan
    r_bad, r_ok = gpu_all(bad, x2), gpu_all(x1, x2)
    keep = [0, 1, 3]
    for k in ("rl", "rr", "match", "cost", "g1", "g2"):
        assert np.array_equal(r_bad[k][keep], r_ok[k][keep]), k
    _, _, mt = cpu_emd.match(bad[2:3], x2[2:3])
    assert np.array_equal(np.isnan(r_bad["match"][2:3]), np.isnan(mt))
    assert np.isnan(r_bad["cost"][2]) and np.isnan(cpu_emd.cost(bad[2:3], x2[2:3], mt)[0])


class _ReferenceStyleEMD(torch.autograd.Function):
    """the reference's extensions/emd autograd Function, written over the emd_cuda module"""

    @staticmethod
    def forward(ctx, xyz1, xyz2):
        import emd_cuda
        xyz1, xyz2 = xyz1.contiguous(), xyz2.contiguous()
        match = emd_cuda.approxmatch_forward(xyz1, xyz2)
        cost = emd_cuda.matchcost_forward(xyz1, xyz2, match)
        ctx.save_for_backward(xyz1, xyz2, match)
        return cost

    @staticmethod
    def backward(ctx, grad_cost):
        import emd_cuda
        xyz1, xyz2, match = ctx.saved_tensors
        grad_xyz1, grad_xyz2 = emd_cuda.matchcost_backward(grad_cost.contiguous(), xyz1, xyz2, match)
        return grad_xyz1, grad_xyz2


def test_drop_in_module():
    import pointdae_b200
    pointdae_b200.install()
    import emd_cuda
    x1 = torch.from_numpy(ball(3, 700, 16)).to(DEV)
    x2 = torch.from_numpy(ball(3, 900, 17)).to(DEV)
    _, _, want = ops.emd_match(x1, x2, materialize=True)
    match = emd_cuda.approxmatch_forward(x1, x2)
    assert match.shape == (3, 900, 700) and match.dtype == torch.float32 and torch.equal(match, want)
    cost = emd_cuda.matchcost_forward(x1, x2, match)
    assert torch.equal(cost, ops.emd_cost(x1, x2, match=want))
    gc = torch.tensor([1.0, 0.5, 2.0], device=DEV)
    g = emd_cuda.matchcost_backward(gc, x1, x2, match)
    assert isinstance(g, list) and all(torch.equal(a, b_) for a, b_ in zip(g, ops.emd_cost_grad(gc, x1, x2, match=want)))
    # the reference-style Function over emd_cuda and the ratio-path Function agree bit for bit
    a1, a2 = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    b1, b2 = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    ca = _ReferenceStyleEMD.apply(a1, a2)
    cb = emd.earth_mover_distance(b1, b2)
    (ca * gc).sum().backward()
    (cb * gc).sum().backward()
    assert torch.equal(ca, cb) and torch.equal(a1.grad, b1.grad) and torch.equal(a2.grad, b2.grad)


def test_cuda_graph_replay_equals_eager():
    x1 = torch.from_numpy(ball(4, 1024, 18)).to(DEV)
    x2 = torch.from_numpy(ball(4, 1024, 19)).to(DEV)
    gc = torch.ones(4, device=DEV)

    def step():
        rl, rr, _ = ops.emd_match(x1, x2)
        cost = ops.emd_cost(x1, x2, ratio_l=rl, ratio_r=rr)
        g1, g2 = ops.emd_cost_grad(gc, x1, x2, ratio_l=rl, ratio_r=rr)
        return cost, g1, g2

    eager = step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = step()
    graph.replay()
    torch.cuda.synchronize()
    for a, b_ in zip(eager, out):
        assert torch.equal(a, b_)
