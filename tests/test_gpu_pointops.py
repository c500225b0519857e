"""Segment FPS / kNN on the GPU (csrc/pointops.cu) against the fp32 oracle (oracle/pdae_oracle_pointops.c), bit for
bit: ragged batches with empty, 1-point and short segments, `n` around the tie-rule and capacity boundaries, every FPS
form, ties, b = 1 and b = 4096.  Also bit-identity across repeats, concurrent streams and CUDA-graph replay,
cross-checks against the equal-size ops and float64 cdist, and the reference's autograd Functions on `pointops_cuda`."""
import numpy as np
import pytest
import torch

from oracle import cpu_pointops as cp
from pointdae_b200 import ops, pointops

pytestmark = pytest.mark.gpu
DEV = "cuda"


def packed(sizes, seed, grid=None, dup=False):
    rng = np.random.default_rng(seed)
    n = int(sum(sizes))
    if grid:
        x = rng.integers(0, grid, (n, 3)).astype(np.float32) * 0.25
    else:
        x = rng.random((n, 3)).astype(np.float32)
    if dup and n > 1:
        x[1::3] = x[0::3][: len(x[1::3])]  # every third point has a twin
    return x, np.cumsum(sizes).astype(np.int32)


def sample_offsets(sizes, frac, minimum=1):
    return np.cumsum([max(minimum, int(s * frac)) for s in sizes]).astype(np.int32)


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def gpu_fps(x, off, noff, n, with_tmp=True):
    m = int(noff[-1])
    idx = torch.full((m,), -7, dtype=torch.int32, device=DEV)
    tmp = torch.full((len(x),), 1e10, dtype=torch.float32, device=DEV) if with_tmp else None
    ops.segment_fps_into(t(x), t(off), t(noff), n, idx, tmp)
    return idx.cpu().numpy(), (tmp.cpu().numpy() if with_tmp else None)


CASES = {
    "ragged": ([100, 0, 1, 300, 7, 0, 2, 31], 0.3, None),
    "n1023": ([1023, 400, 1], 0.1, None),
    "n1024": ([1024, 1000, 0], 0.1, None),
    "n1025": ([1025, 17], 0.1, None),
    "reg2048": ([2048, 1500, 33], 0.05, None),
    "global20k": ([20000, 3000], 0.01, None),
    "global250k": ([250000, 100], 0.0004, None),
    "n_below_largest": ([9000, 300, 20000], 0.01, 512),   # register form chosen from n, segments above its capacity
    "b1": ([3000], 0.1, None),
    "b4096": (list(np.random.default_rng(0).integers(0, 40, 4096)), 0.25, None),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("kind", ["random", "grid", "dup"])
def test_fps_matches_oracle(case, kind):
    sizes, frac, n = CASES[case]
    if kind != "random" and case in ("global250k", "b4096"):
        pytest.skip("one input kind is enough at this size")
    x, off = packed(sizes, 11, grid=6 if kind == "grid" else None, dup=kind == "dup")
    noff = sample_offsets(sizes, frac)
    n = cp.largest(off) if n is None else n
    want_i, want_t = cp.seg_fps(x, off, noff, n=n, tmp=np.full(len(x), 1e10, np.float32))
    got_i, got_t = gpu_fps(x, off, noff, n)
    assert np.array_equal(got_i, want_i)
    assert np.array_equal(got_t.view(np.uint32), want_t.view(np.uint32))
    assert np.array_equal(gpu_fps(x, off, noff, n, with_tmp=False)[0], want_i)


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("nsample", [1, 16, 33, 100])
def test_knn_matches_oracle(case, nsample):
    sizes, frac, _ = CASES[case]
    if case == "global250k" and nsample != 16:
        pytest.skip("one nsample is enough at this size")
    x, off = packed(sizes, 12, grid=6 if nsample == 33 else None, dup=nsample == 100)
    q, qoff = packed([max(1, int(s * frac)) for s in sizes], 13)
    qx = np.concatenate([q, np.random.default_rng(1).random((5, 3)).astype(np.float32)])  # 5 rows past the last segment
    want_i, want_d = cp.seg_knn(nsample, x, qx, off, qoff)
    got_i, got_d = ops.segment_knn(nsample, t(x), t(qx), t(off), t(qoff))
    assert np.array_equal(got_i.cpu().numpy(), want_i)
    assert np.array_equal(got_d.cpu().numpy().view(np.uint32), want_d.view(np.uint32))
    assert (got_i[-5:] == -1).all() and (got_d[-5:] == 1e10).all()


def test_public_functions_and_defaults():
    sizes = [700, 0, 1, 1200, 5]
    x, off = packed(sizes, 14)
    noff = sample_offsets(sizes, 0.1)
    want, _ = cp.seg_fps(x, off, noff)
    assert np.array_equal(pointops.furthestsampling(t(x), t(off), t(noff)).cpu().numpy(), want)
    assert np.array_equal(ops.segment_fps(t(x), t(off), t(noff), n=cp.largest(off), m=int(noff[-1])).cpu().numpy(), want)
    wi, wd = cp.seg_knn(8, x, x, off, off)
    gi, gd = pointops.knnquery(8, t(x), None, t(off), t(off))
    assert np.array_equal(gi.cpu().numpy(), wi) and torch.equal(gd, torch.sqrt(t(wd)))


def test_repeat_streams_and_graph():
    sizes = [5000, 300, 0, 12000, 900]
    x, off = packed(sizes, 15)
    noff = sample_offsets(sizes, 0.05)
    X, O, N = t(x), t(off), t(noff)
    n, m = cp.largest(off), int(noff[-1])
    ref_i = ops.segment_fps(X, O, N, n=n, m=m)
    ref_k = ops.segment_knn(16, X, X[ref_i.long()], O, N)
    for _ in range(3):
        assert torch.equal(ops.segment_fps(X, O, N, n=n, m=m), ref_i)
        k = ops.segment_knn(16, X, X[ref_i.long()], O, N)
        assert torch.equal(k[0], ref_k[0]) and torch.equal(k[1], ref_k[1])
    # two streams at once
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    outs = []
    for s in (s1, s2):
        with torch.cuda.stream(s):
            outs.append((ops.segment_fps(X, O, N, n=n, m=m), ops.segment_knn(16, X, X, O, O)))
    torch.cuda.synchronize()
    assert torch.equal(outs[0][0], ref_i) and torch.equal(outs[1][0], ref_i)
    assert torch.equal(outs[0][1][0], outs[1][1][0]) and torch.equal(outs[0][1][1], outs[1][1][1])
    # CUDA-graph capture of the drop-in module's calls, replayed on new contents of the same buffers
    from pointdae_b200 import pointops_cuda
    idx = torch.zeros(m, dtype=torch.int32, device=DEV)
    tmp = torch.empty(len(x), device=DEV)
    q = torch.empty((m, 3), device=DEV)
    ki = torch.zeros((m, 16), dtype=torch.int32, device=DEV)
    kd = torch.zeros((m, 16), device=DEV)
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        tmp.fill_(1e10)  # warm-up outside the capture
        pointops_cuda.furthestsampling_cuda(len(sizes), n, X, O, N, tmp, idx)
        torch.cuda.synchronize()
        with torch.cuda.graph(g, stream=s):
            tmp.fill_(1e10)
            pointops_cuda.furthestsampling_cuda(len(sizes), n, X, O, N, tmp, idx)
            torch.index_select(X, 0, idx.long(), out=q)
            pointops_cuda.knnquery_cuda(m, 16, X, q, O, N, ki, kd)
    torch.cuda.current_stream().wait_stream(s)
    for seed in (16, 17):
        x2, _ = packed(sizes, seed)
        X.copy_(t(x2))
        g.replay()
        torch.cuda.synchronize()
        wi, wt = cp.seg_fps(x2, off, noff, tmp=np.full(len(x2), 1e10, np.float32))
        wki, wkd = cp.seg_knn(16, x2, x2[wi], off, noff)
        assert np.array_equal(idx.cpu().numpy(), wi) and np.array_equal(tmp.cpu().numpy(), wt)
        assert np.array_equal(ki.cpu().numpy(), wki) and np.array_equal(kd.cpu().numpy(), wkd)


@pytest.mark.parametrize("b,n,npoint", [(16, 1000, 128), (4, 512, 64), (32, 129, 32)])
def test_fps_equals_equal_size_op(b, n, npoint):
    # no point within |p|^2 <= 1e-3 of the origin, where pointnet2's FPS skips points and pointops does not
    rng = np.random.default_rng(b + n)
    x = rng.uniform(0.1, 1.0, (b, n, 3)).astype(np.float32)
    want = ops.furthest_point_sample(t(x), npoint).cpu().numpy() + (np.arange(b) * n)[:, None]
    off = (np.arange(1, b + 1) * n).astype(np.int32)
    noff = (np.arange(1, b + 1) * npoint).astype(np.int32)
    got = ops.segment_fps(t(x.reshape(-1, 3)), t(off), t(noff)).cpu().numpy()
    assert np.array_equal(got, want.reshape(-1))


@pytest.mark.parametrize("b,n,q,k", [(8, 2048, 256, 32), (128, 512, 64, 16), (3, 5000, 700, 100)])
def test_knn_equals_equal_size_op_and_cdist(b, n, q, k):
    rng = np.random.default_rng(b * k)
    x = rng.standard_normal((b, n, 3)).astype(np.float32)
    qx = rng.standard_normal((b, q, 3)).astype(np.float32)
    _, want = ops.knn_points(t(x), t(qx), k)
    want = want.cpu().numpy() + (np.arange(b) * n)[:, None, None]
    off = (np.arange(1, b + 1) * n).astype(np.int32)
    qoff = (np.arange(1, b + 1) * q).astype(np.int32)
    gi, gd = ops.segment_knn(k, t(x.reshape(-1, 3)), t(qx.reshape(-1, 3)), t(off), t(qoff))
    gi = gi.cpu().numpy()
    assert np.array_equal(gi, want.reshape(-1, k))
    # float64 neighbour sets: equal wherever the k-th and (k+1)-th float64 distances are apart
    d = torch.cdist(t(qx).double(), t(x).double()) ** 2
    top = torch.topk(d, k + 1, dim=-1, largest=False)
    sep = (top.values[..., k] - top.values[..., k - 1]).cpu().numpy().reshape(-1) > 1e-5
    sets = np.sort(top.indices[..., :k].cpu().numpy() + (np.arange(b) * n)[:, None, None], -1).reshape(-1, k)
    assert sep.mean() > 0.99
    assert np.array_equal(np.sort(gi, -1)[sep], sets[sep])


# the reference's autograd Functions (PointTransformer lib/pointops/functions/pointops.py), verbatim but for the import
REFERENCE_FUNCTIONS = '''
from torch.autograd import Function
import pointops_cuda


class FurthestSampling(Function):
    @staticmethod
    def forward(ctx, xyz, offset, new_offset):
        """
        input: xyz: (n, 3), offset: (b), new_offset: (b)
        output: idx: (m)
        """
        assert xyz.is_contiguous()
        n, b, n_max = xyz.shape[0], offset.shape[0], offset[0]
        for i in range(1, b):
            n_max = max(offset[i] - offset[i-1], n_max)
        idx = torch.cuda.IntTensor(new_offset[b-1].item()).zero_()
        tmp = torch.cuda.FloatTensor(n).fill_(1e10)
        pointops_cuda.furthestsampling_cuda(b, n_max, xyz, offset, new_offset, tmp, idx)
        del tmp
        return idx

furthestsampling = FurthestSampling.apply


class KNNQuery(Function):
    @staticmethod
    def forward(ctx, nsample, xyz, new_xyz, offset, new_offset):
        """
        input: xyz: (n, 3), new_xyz: (m, 3), offset: (b), new_offset: (b)
        output: idx: (m, nsample), dist2: (m, nsample)
        """
        if new_xyz is None: new_xyz = xyz
        assert xyz.is_contiguous() and new_xyz.is_contiguous()
        m = new_xyz.shape[0]
        idx = torch.cuda.IntTensor(m, nsample).zero_()
        dist2 = torch.cuda.FloatTensor(m, nsample).zero_()
        pointops_cuda.knnquery_cuda(m, nsample, xyz, new_xyz, offset, new_offset, idx, dist2)
        return idx, torch.sqrt(dist2)

knnquery = KNNQuery.apply
'''


def test_reference_functions_run_on_the_drop_in():
    import sys
    import pointdae_b200
    saved = sys.modules.get("pointops_cuda")
    try:
        pointdae_b200.install()
        ns = {"torch": torch}
        exec(compile(REFERENCE_FUNCTIONS, "pointops_reference_functions", "exec"), ns)
        sizes = [900, 0, 1, 1500, 40]
        x, off = packed(sizes, 18)
        noff = sample_offsets(sizes, 0.1)
        X = t(x).requires_grad_(True)
        idx = ns["furthestsampling"](X, t(off), t(noff))
        want_i, _ = cp.seg_fps(x, off, noff)
        assert np.array_equal(idx.cpu().numpy(), want_i)
        ki, kd = ns["knnquery"](16, X, X[idx.long()].detach().contiguous(), t(off), t(noff))
        wki, wkd = cp.seg_knn(16, x, x[want_i], off, noff)
        assert np.array_equal(ki.cpu().numpy(), wki) and torch.equal(kd, torch.sqrt(t(wkd)))
    finally:
        if saved is None:
            sys.modules.pop("pointops_cuda", None)
        else:
            sys.modules["pointops_cuda"] = saved
