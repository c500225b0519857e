"""The FP32-pipe Chamfer forward (csrc/chamfer.cu, scan body in chamfer_core.cuh) in every form the library selects:
symmetric with the list column recovery (up to 128 row groups of 128 rows) or the warp-per-column recovery (larger
clouds), the two-scan path, and column-split units (every 512-row block's sweep cut into column chunks whose row minima
merge through packed (distance, index) keys).  Results must not depend on the form, the chunk count, the phased entry
point or the workspace size the caller offers -- and must equal the oracle (chamfer.cu:15-171 restated).

The tensor-core filter (chamfer_tc.cu) serves clouds of at least 512 points by default, so every test here pins the
FP32-pipe forward and runs its cases again under the library default: the shapes the filter takes keep their checks
on that path too."""
import numpy as np
import pytest
import torch

from oracle import cpu as oracle
from pointdae_b200 import _native, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture
def modes():
    """Pins the FP32-pipe forward (pdae_tune_chamfer_tc mode 0) for the test and restores the previous mode afterwards.
    Yields `modes()`: iterating it runs the loop body in mode 0, then in the library default, and ends in mode 0."""
    L = _native.lib()
    default = L.pdae_tune_chamfer_tc(0, 0.0)
    assert L.pdae_tune_chamfer_tc(-1, 0.0) == 0, "the FP32-pipe forward could not be pinned"

    def each():
        for mode in (0,) if default == 0 else (0, default):
            L.pdae_tune_chamfer_tc(mode, 0.0)
            assert L.pdae_tune_chamfer_tc(-1, 0.0) == mode
            yield mode
        L.pdae_tune_chamfer_tc(0, 0.0)

    yield each
    L.pdae_tune_chamfer_tc(default, 0.0)


@pytest.fixture
def split_hook():
    L = _native.lib()
    old = L.pdae_tune_chamfer_split(-1)
    yield L.pdae_tune_chamfer_split
    L.pdae_tune_chamfer_split(old)


def assert_equals_oracle(got, want, what):
    for g, w, name in zip(got, want, ("dist1", "dist2", "idx1", "idx2")):
        np.testing.assert_array_equal(g.cpu().numpy(), w, err_msg="%s, %s" % (name, what))


# (1, 16384, 9000): 128 row groups, the most the list recovery serves; (2, 16385, 700) and (1, 20000, 3000): above
# that, the warp-per-column recovery; (6, 250, 140): clouds up to 256 points take the one-query-per-thread two-scan
# kernel whatever the caller asks for.
@pytest.mark.parametrize("b,n,m", [(3, 700, 1300), (37, 2048, 2048), (2, 129, 4097), (5, 513, 257), (1, 16384, 9000),
                                   (300, 260, 300), (2, 16385, 700), (1, 20000, 3000), (6, 250, 140)])
def test_chamfer_fp32_forms_agree_bit_for_bit(modes, split_hook, b, n, m):
    """symmetric unsplit, split into 3 chunks, automatic split, with a column-key-only workspace, and two-scan: each
    equals the oracle bit for bit (hence each other) on ragged, tied and multi-pass shapes."""
    x1 = cu(synth.adversarial(synth.clouds(b, n, seed=600 + n), seed=n, n_small=0, n_dup=min(40, n // 4)))
    x2 = cu(synth.adversarial(synth.clouds(b, m, seed=700 + m), seed=m, n_small=0, n_dup=min(40, m // 4)))
    x2[:, : min(n, m) // 2] = x1[:, : min(n, m) // 2]  # exact zeros and cross-cloud ties
    want = oracle.chamfer_fwd(x1.cpu().numpy(), x2.cpu().numpy())
    for mode in modes():
        for nc in (1, 3, 0):
            split_hook(nc)
            assert_equals_oracle(ops.chamfer_forward(x1, x2), want, "symmetric, split hook %d, mode %d" % (nc, mode))
        with ops.chamfer_column_split(False):
            assert_equals_oracle(ops.chamfer_forward(x1, x2), want, "column keys only, mode %d" % mode)
        assert_equals_oracle(ops.chamfer_forward(x1, x2, symmetric=False), want, "two-scan, mode %d" % mode)


@pytest.mark.parametrize("b,n,m", [(2, 2048, 2048), (3, 700, 1300), (2, 1300, 700), (1, 5000, 300), (2, 300, 5000), (4, 513, 257)])
def test_chamfer_symmetric_and_two_pass_kernels_agree(modes, b, n, m):
    """The single-evaluation (workspace) path and the two-scan path must give identical bits."""
    x1 = cu(synth.adversarial(synth.clouds(b, n, seed=700 + n), seed=n, n_small=0, n_dup=n // 8))
    x2 = cu(synth.adversarial(synth.clouds(b, m, seed=800 + m), seed=m, n_small=0, n_dup=m // 8))
    x2[:, : min(n, m) // 2] = x1[:, : min(n, m) // 2]  # exact zero distances and cross-cloud ties
    wd1, wd2, wi1, wi2 = oracle.chamfer_fwd(x1.cpu().numpy(), x2.cpu().numpy())
    for mode in modes():
        a = ops.chamfer_forward(x1, x2, symmetric=True)
        c = ops.chamfer_forward(x1, x2, symmetric=False)
        for u, v in zip(a, c):
            assert torch.equal(u, v), mode
        np.testing.assert_array_equal(a[2].cpu().numpy(), wi1)
        np.testing.assert_array_equal(a[3].cpu().numpy(), wi2)
        np.testing.assert_array_equal(a[1].cpu().numpy(), wd2)


@pytest.mark.parametrize("b,n,m", [(1, 2048, 2048), (3, 1500, 700), (2, 513, 1025), (5, 300, 2049), (2, 4096, 4095),
                                   (7, 1024, 1024), (1, 20000, 3000)])
def test_every_chunk_count_equals_the_oracle(modes, split_hook, b, n, m):
    a, c = synth.clouds(b, n, seed=n + b), synth.clouds(b, m, seed=m + 7)
    a[:, 5] = c[:, 3]          # exact zero distance
    c[:, 11] = c[:, 10]        # duplicate reference point: the lower index must win in every chunking
    if m > 700:
        c[:, 600] = c[:, 10]   # ... also across chunk / tile boundaries
        a[:, 9] = a[:, 8]
    want = oracle.chamfer_fwd(a, c)
    ta, tc = cu(a), cu(c)
    for mode in modes():
        for nc in (1, 2, 3, 5, 16, 0):
            split_hook(nc)
            assert_equals_oracle(ops.chamfer_forward(ta, tc), want, "%d chunks, mode %d" % (nc, mode))


def test_headline_shape_split_vs_unsplit_and_context_manager(modes, split_hook):
    a = cu(synth.prediction(synth.clouds(128, 2048, seed=1), seed=1))
    c = cu(synth.clouds(128, 2048, seed=1))
    for mode in modes():
        split_hook(1)
        want = ops.chamfer_forward(a, c)
        for nc in (0, 2, 4):
            split_hook(nc)
            got = ops.chamfer_forward(a, c)
            assert all(torch.equal(g, w) for g, w in zip(got, want)), (nc, mode)
        split_hook(2)
        with ops.chamfer_column_split(False):  # column-key-only workspace: the library cannot split
            got = ops.chamfer_forward(a, c)
        assert all(torch.equal(g, w) for g, w in zip(got, want)), mode
        ev = torch.cuda.Event()
        got = ops.chamfer_forward(a, c, scan_done=ev)  # phased entry point: separate unpack launch, same values
        assert all(torch.equal(g, w) for g, w in zip(got, want)), mode


def test_split_forward_feeds_the_fused_loss_and_backward(modes, split_hook):
    from pointdae_b200 import chamfer_dist
    xyz = synth.clouds(4, 3000, seed=3)
    pred = synth.prediction(xyz, seed=3)
    for mode in modes():
        outs = []
        for nc in (1, 3):
            split_hook(nc)
            p = cu(pred).requires_grad_(True)
            loss = chamfer_dist.ChamferDistanceL1()(p, cu(xyz))
            loss.backward()
            outs.append((loss.detach().clone(), p.grad.clone()))
        assert torch.equal(outs[0][0], outs[1][0]), mode
        assert torch.allclose(outs[0][1], outs[1][1], rtol=1e-6, atol=1e-9), mode  # atomics: order-free sums


@pytest.mark.parametrize("n,m,lo,hi", [(3000, 5000, 1000, 3600), (100000, 30000, 0, 12500), (700, 2000, 1999, 2000)])
def test_sharded_entry_points_merge_their_chunks_into_the_returned_keys(modes, split_hook, n, m, lo, hi):
    """pdae_chamfer_sharded_f32 / pdae_chamfer_min_keys_u64: the packed row keys a rank hands to the MIN all-reduce are
    themselves the merge target of its column-split units (global indices, identity-filled first)."""
    a = cu(synth.prediction(synth.clouds(1, max(n, m), seed=n), seed=n)[:, :n])
    c = cu(synth.clouds(1, max(n, m), seed=n)[:, :m])
    c[:, lo + 1 if lo + 1 < hi else lo] = c[:, lo]  # duplicate inside the slice
    sl = c[:, lo:hi].contiguous()
    for mode in modes():
        split_hook(1)
        want = ops.chamfer_sharded_local(a, sl, lo)
        want_keys = ops.chamfer_min_keys(a, sl, lo)
        assert torch.equal(want[0], want_keys)
        d, i = ops.chamfer_unpack_keys(want[0])
        assert int(i.min()) >= lo and int(i.max()) < hi
        for nc in (2, 3, 7, 0):
            split_hook(nc)
            got = ops.chamfer_sharded_local(a, sl, lo)
            assert all(torch.equal(g, w) for g, w in zip(got, want)), (nc, mode)
            assert torch.equal(ops.chamfer_min_keys(a, sl, lo), want_keys), (nc, mode)
