"""Chamfer forward through the tensor-core filter (csrc/chamfer_tc.cu) -- the default for clouds of 512..2048 points --
against the CPU oracle (extensions/chamfer_dist/chamfer.cu:15-145 restated), stored outputs of the reference's own CUDA
kernel, and the FP32-pipe kernels of csrc/chamfer.cu.  Bar: dist and idx bit-exact, for every input: the filter only
decides which 32-column groups are evaluated exactly, never the result."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import cpu as oracle
from pointdae_b200 import _native, chamfer_dist, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CHAMFER_GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "chamfer.npz"))


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture()
def tc_mode():
    """yields a setter for the tuning hook and restores the library default afterwards"""
    lib = _native.lib()
    old = lib.pdae_tune_chamfer_tc(-1, 0.0)

    def set_mode(mode, eps_rel=-1.0):  # eps_rel < 0: the mode's default bound
        lib.pdae_tune_chamfer_tc(mode, eps_rel)

    yield set_mode
    lib.pdae_tune_chamfer_tc(old, -1.0)


def probe(a, b):
    bs, n, m = a.size(0), a.size(1), b.size(1)
    d1, d2 = torch.empty((bs, n), device=DEV), torch.empty((bs, m), device=DEV)
    i1, i2 = torch.empty((bs, n), dtype=torch.int32, device=DEV), torch.empty((bs, m), dtype=torch.int32, device=DEV)
    st = torch.zeros(4, dtype=torch.int64, device=DEV)
    rc = _native.lib().pdae_chamfer_tc_probe(a.data_ptr(), b.data_ptr(), bs, n, m, d1.data_ptr(), d2.data_ptr(), i1.data_ptr(),
                                             i2.data_ptr(), st.data_ptr(), None,
                                             ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    _native.check(rc, "pdae_chamfer_tc_probe")
    s = st.cpu().numpy()
    err = float(np.array([int(s[0]) & 0xffffffff], dtype=np.uint32).view(np.float32)[0])
    return [d1, d2, i1, i2], {"max_rel_err": err, "scan_rows": int(s[1]), "groups": int(s[2]), "rows": int(s[3])}


def clouds_pair(kind, bs, n, m, seed):
    c = synth.clouds(bs, max(n, m), seed=seed)
    rng = np.random.default_rng(seed)
    if kind == "prediction":
        p = synth.prediction(c, seed=seed)
    elif kind == "ties":  # duplicates and an exact permuted copy: every minimum is 0 and attained several times
        c = synth.adversarial(c, seed=seed, n_small=8, n_dup=min(200, max(n, m) // 4))
        p = synth.prediction(c, seed=seed, sigma=0.0)
    elif kind == "lattice":  # coordinates on a coarse lattice: exact ties between distinct points everywhere
        c = rng.integers(0, 12, size=c.shape).astype(np.float32) * np.float32(0.125)
        p = c[:, ::-1].copy()
    elif kind == "blob":  # an untrained decoder: every prediction near the origin
        p = (rng.standard_normal(c.shape) * 0.03).astype(np.float32)
    elif kind == "offset":  # far from the origin: the centring carries the filter's precision
        p = (synth.prediction(c, seed=seed) * 3 + 40).astype(np.float32)
        c = (c * 3 + 40).astype(np.float32)
    else:
        raise ValueError(kind)
    return np.ascontiguousarray(p[:, :n]), np.ascontiguousarray(c[:, :m])


ORACLE_CASES = [
    ("prediction", 3, 1024, 1024), ("prediction", 2, 2048, 2048), ("prediction", 2, 777, 2041), ("prediction", 2, 2048, 513),
    ("ties", 2, 1024, 1024), ("ties", 2, 1536, 640), ("lattice", 2, 1024, 2048), ("lattice", 3, 640, 640),
    ("blob", 2, 2048, 1024), ("offset", 2, 1024, 1024), ("offset", 1, 2047, 1999),
]


@pytest.mark.parametrize("mode", [1, 2, 3])
@pytest.mark.parametrize("kind,bs,n,m", ORACLE_CASES)
def test_tc_forward_matches_oracle(tc_mode, mode, kind, bs, n, m):
    tc_mode(mode)
    a, b = clouds_pair(kind, bs, n, m, seed=n + m)
    want = oracle.chamfer_fwd(a, b)
    got = ops.chamfer_forward(cu(a), cu(b))
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g.cpu().numpy(), w)


@pytest.mark.parametrize("kind", ["prediction", "ties", "lattice", "blob", "offset"])
@pytest.mark.parametrize("bs,n,m", [(128, 2048, 2048), (128, 1024, 1024), (40, 1536, 2048), (300, 512, 640)])
def test_tc_forward_equals_the_fp32_pipe_kernels_at_full_size(tc_mode, kind, bs, n, m):
    base_a, base_b = clouds_pair(kind, min(bs, 16), n, m, seed=7 * n + m)
    reps = -(-bs // base_a.shape[0])
    a = cu(np.tile(base_a, (reps, 1, 1))[:bs])
    b = cu(np.tile(base_b, (reps, 1, 1))[:bs])
    if kind == "prediction":  # distinct clouds, not tiles of sixteen
        a = a + 1e-3 * torch.randn(a.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(n))
    tc_mode(0)
    want = ops.chamfer_forward(a, b)
    for mode in (3, 2, 1):
        tc_mode(mode)
        got = ops.chamfer_forward(a, b)
        assert all(torch.equal(g, w) for g, w in zip(got, want)), (mode, kind)


CHUNKED = [("prediction", 2, 4096, 4096), ("ties", 1, 8192, 3000), ("prediction", 2, 2049, 5000), ("lattice", 1, 20000, 777),
           ("offset", 1, 6000, 6000), ("blob", 3, 1000, 4100)]


@pytest.mark.parametrize("mode", [2, 3])
@pytest.mark.parametrize("kind,bs,n,m", CHUNKED)
def test_tc_forward_in_column_chunks_matches_oracle(tc_mode, mode, kind, bs, n, m):
    """clouds above 2048 points: the searched cloud is cut into column chunks whose (distance, index) keys merge with
    RED.MIN in the forward's workspace -- same bits as the oracle, lowest index on ties across chunk boundaries"""
    tc_mode(mode)
    a, b = clouds_pair(kind, bs, n, m, seed=n + m)
    want = oracle.chamfer_fwd(a, b)
    got = ops.chamfer_forward(cu(a), cu(b))
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g.cpu().numpy(), w)


@pytest.mark.parametrize("bs,n,m", [(16, 8192, 8192), (1, 100000, 100000), (2, 30000, 2048)])
def test_tc_forward_in_column_chunks_equals_the_fp32_pipe_kernels(tc_mode, bs, n, m):
    a, b = clouds_pair("prediction", bs, n, m, seed=n)
    ta, tb = cu(a), cu(b)
    tc_mode(0)
    want = ops.chamfer_forward(ta, tb)
    for mode in (3, 2):
        tc_mode(mode)
        got = ops.chamfer_forward(ta, tb)
        assert all(torch.equal(g, w) for g, w in zip(got, want)), mode


@pytest.mark.parametrize("mode", [0, 2, 3])
@pytest.mark.parametrize("n,m,world", [(100000, 100000, 8), (5000, 3000, 3), (1500, 40000, 5)])
def test_reference_set_sharded_share_through_the_tensor_cores(tc_mode, mode, n, m, world):
    """pdae_chamfer_sharded_f32 rank by rank in one process (SURVEY.md 8e): MIN over the ranks' row keys and the slices'
    final column results equal the unsharded forward, whichever kernel family serves the rank's share"""
    a, b = clouds_pair("prediction", 1, n, m, seed=n + world)
    t1, t2 = cu(a), cu(b)
    tc_mode(0)
    d1, d2, i1, i2 = ops.chamfer_forward(t1, t2)
    tc_mode(mode)
    keys = None
    for r in range(world):
        lo, hi = r * m // world, (r + 1) * m // world
        k, d2l, i2l = ops.chamfer_sharded_local(t1, t2[:, lo:hi].contiguous(), lo)
        keys = k if keys is None else torch.minimum(keys, k)
        assert torch.equal(d2l, d2[:, lo:hi]) and torch.equal(i2l, i2[:, lo:hi]), r
    sd, si = ops.chamfer_unpack_keys(keys)
    assert torch.equal(sd, d1) and torch.equal(si, i1)


@pytest.mark.parametrize("case", sorted({k.split("/")[0] for k in CHAMFER_GOLD.files if "/" in k} - {"transposed"}))
def test_fp32_pipe_kernels_still_match_reference_cuda(tc_mode, case):
    """the FP32-pipe kernels (mode 0: every shape outside the tensor-core range, the sharded entry points) and both
    tensor-core modes give what the reference's own chamfer.forward returned on a B200 (chamfer.npz), bit for bit"""
    z = CHAMFER_GOLD
    x1, x2 = cu(z[case + "/xyz1"]), cu(z[case + "/xyz2"])
    for mode in (0, 2, 3):
        tc_mode(mode)
        got = ops.chamfer_forward(x1, x2)
        for g, key in zip(got, ("dist1", "dist2", "idx1", "idx2")):
            np.testing.assert_array_equal(g.cpu().numpy(), z[case + "/" + key], err_msg="mode %d %s" % (mode, key))


@pytest.mark.parametrize("mode", [2, 3])
def test_tc_mass_ties_take_the_full_scan_and_stay_exact(tc_mode, mode):
    """every point identical (and a cloud of only two distinct points): every group ties, the candidate lists overflow and
    the rows are decided by the exact scan over all columns -- lowest index, like the reference's strict `<`"""
    tc_mode(mode)
    a = np.zeros((2, 1024, 3), dtype=np.float32)
    b = np.zeros((2, 2048, 3), dtype=np.float32)
    a[0] += np.float32(0.25)
    b[0] += np.float32(0.25)
    a[1, ::2] = (0.5, -0.25, 0.125)
    b[1, 1::3] = (0.5, -0.25, 0.125)
    want = oracle.chamfer_fwd(a, b)
    got, st = probe(cu(a), cu(b))
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g.cpu().numpy(), w)
    assert st["scan_rows"] > 0
    assert (got[2].cpu().numpy()[0] == 0).all() and (got[3].cpu().numpy()[0] == 0).all()


@pytest.mark.parametrize("mode", [2, 3])
def test_tc_non_finite_and_huge_coordinates_fall_back_to_the_literal_scan(tc_mode, mode):
    """a NaN, an infinity, or coordinates too large for the filter's bound: the cloud is scanned literally
    (`k == 0 || d < best`, chamfer.cu:47-79) -- the oracle's semantics"""
    tc_mode(mode)
    a, b = clouds_pair("prediction", 4, 1024, 1024, seed=3)
    b[0, 5, 1] = np.nan
    a[1, 17, 0] = np.inf
    a[2] *= np.float32(3e15)
    b[2] *= np.float32(3e15)
    want = oracle.chamfer_fwd(a, b)
    got = ops.chamfer_forward(cu(a), cu(b))
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g.cpu().numpy(), w)


@pytest.mark.parametrize("mode,tight", [(2, 2.0 ** -23), (3, 2.0 ** -21)])
def test_tc_filter_error_and_margin(tc_mode, mode, tight):
    """the observed error of the approximate group minima stays 8x under the default bound (2^-17 / 2^-16 of the scale), the
    result does not change with a bound 32-64x tighter, and about one group per row is evaluated exactly"""
    a, b = clouds_pair("prediction", 32, 2048, 2048, seed=11)
    ta, tb = cu(a), cu(b)
    tc_mode(0)
    want = ops.chamfer_forward(ta, tb)
    tc_mode(mode)
    got, st = probe(ta, tb)
    assert all(torch.equal(g, w) for g, w in zip(got, want))
    assert st["max_rel_err"] < 2.0 ** -20, st
    assert st["rows"] == 2 * 32 * 2048 and st["groups"] <= st["rows"], st
    tc_mode(mode, tight)
    got, st = probe(ta, tb)
    assert all(torch.equal(g, w) for g, w in zip(got, want))


def test_public_modules_run_on_the_tensor_core_path(tc_mode):
    """ChamferDistanceL2 / ChamferFunction (extensions/chamfer_dist/__init__.py:31-50) with the default mode: same loss and
    gradient as with the FP32-pipe kernels"""
    a, b = clouds_pair("prediction", 6, 2048, 2048, seed=21)
    out = {}
    for mode in (0, 3):
        tc_mode(mode)
        p = cu(a).requires_grad_(True)
        loss = chamfer_dist.ChamferDistanceL2()(p, cu(b))
        loss.backward()
        out[mode] = (float(loss.detach()), p.grad.clone())
    assert out[0][0] == out[3][0]
    assert torch.allclose(out[0][1], out[3][1], rtol=1e-5, atol=1e-5 * float(out[0][1].abs().max()))
