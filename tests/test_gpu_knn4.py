"""Second-generation 3-D kNN / Group kernel (csrc/knn4.cu): every schedule it can take -- the four (queries per warp,
warps per CTA, warp-specialised) forms, TMA on / off, small tiles (many tiles on small clouds), chunks along the
reference cloud + merge -- gives the oracle's result bit for bit, including clouds whose rows are not 16-byte aligned
(register staging), mass ties (the exact warp-select fallback), k up to 64, the planar DGCNN entry point and the fused
corruption epilogue.  The schedule is forced through pdae_tune_knn; the product picks it automatically.  Clouds too long
for one chunk's step numbers go to the streaming warp-select of csrc/knn.cu, also checked here."""
import itertools

import numpy as np
import pytest
import torch

import _oracle_ops
from oracle import cpu as oracle
from pointdae_b200 import _native, group, knn_cuda, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture
def tune():
    L = _native.lib()

    def set_(form=-1, tile=-1, nz=-1, tma=-1):
        assert L.pdae_tune_knn(form, tile, nz, tma) == 0
    yield set_
    assert L.pdae_tune_knn(-1, -1, -1, -1) == 0


# form: 0 = 4 queries per warp, 8 warps, warp-specialised; 1 = (4, 8); 2 = (4, 4); 3 = (2, 4)
SCHEDULES = [dict(form=form, tile=tile, nz=nz, tma=tma)
             for form, tile, nz, tma in itertools.product(range(4), (256, 1024), (1, 3), (0, 1))]


@pytest.mark.parametrize("r,q,k,adv", [(3000, 70, 32, True), (2999, 33, 20, True), (5000, 40, 64, False), (777, 29, 5, True)])
def test_every_schedule_matches_the_oracle(tune, r, q, k, adv):
    b = 2
    ref = synth.clouds(b, r, seed=40 + r)
    if adv:
        ref = synth.adversarial(ref, seed=r, n_small=0, n_dup=min(48, r // 4))
    rng = np.random.default_rng(r)
    query = np.take_along_axis(ref, rng.integers(0, r, size=(b, q))[:, :, None], axis=1).copy()
    query[:, ::2] += np.float32(0.01)
    wd, wi = oracle.knn(ref, query, k)
    R, Q = cu(ref), cu(query)
    for cfg in SCHEDULES:
        tune(**cfg)
        D, I = ops.knn_points(R, Q, k)
        assert torch.equal(I.cpu(), torch.from_numpy(wi)), cfg
        assert torch.equal(D.cpu(), torch.from_numpy(wd)), cfg


def test_mass_ties_take_the_exact_fallback_in_every_schedule(tune):
    """200 copies of one point around every query: the candidate queue (64 keys) overflows, the query is redone by the
    streaming warp-select; the tie order must still be 'lower index first'."""
    b, r, q, k = 2, 2600, 24, 32
    ref = synth.clouds(b, r, seed=5)
    ref[:, 100:300] = ref[:, 7:8]          # 200 duplicates of point 7
    ref[:, 1500:1560] = ref[:, 9:10]
    query = ref[:, [7, 9, 11] * 8].copy()
    wd, wi = oracle.knn(ref, query, k)
    R, Q = cu(ref), cu(query)
    for cfg in SCHEDULES:
        tune(**cfg)
        D, I = ops.knn_points(R, Q, k)
        assert torch.equal(I.cpu(), torch.from_numpy(wi)), cfg
        assert torch.equal(D.cpu(), torch.from_numpy(wd)), cfg


@pytest.mark.parametrize("n,k", [(2600, 20), (1027, 7)])
def test_planar_self_knn_every_schedule(tune, n, k):
    """DGCNN layer 1 (C = 3): x (B,3,N) planar, every point a query."""
    x = np.ascontiguousarray(synth.adversarial(synth.clouds(2, n, seed=n), seed=n, n_small=0, n_dup=16).transpose(0, 2, 1))
    want, _ = oracle.feat_knn(x, k)
    X = cu(x)
    for cfg in SCHEDULES:
        tune(**cfg)
        got = ops.feat_knn(X, k)
        assert torch.equal(got.cpu(), torch.from_numpy(want)), cfg


def test_group_and_corruption_epilogues_every_schedule(tune):
    b, n, g, m = 2, 3000, 40, 32
    xyz = synth.adversarial(synth.clouds(b, n, seed=77), seed=3)
    want_nb, want_c, want_idx, _ = oracle.group(xyz, g, m)
    X = cu(xyz)
    C = cu(want_c)
    mats_cpu = torch.from_numpy(np.random.default_rng(1).standard_normal((b, 2, 3, 3)).astype(np.float32))
    mats = mats_cpu.to(DEV)
    want_aff = _oracle_ops.group_affine(torch.from_numpy(xyz), torch.from_numpy(want_c), m, mats_cpu, want_idx=True)
    for cfg in SCHEDULES:
        tune(**cfg)
        nb, idx = ops.group_points_knn(X, C, m, want_idx=True)
        assert torch.equal(idx.cpu(), torch.from_numpy(want_idx)), cfg
        assert torch.equal(nb.cpu(), torch.from_numpy(want_nb)), cfg
        got_aff = ops.group_affine(X, C, m, mats, want_idx=True)
        for a, w in zip(got_aff, want_aff):  # neighbourhood, corrupted neighbourhood, corrupted centre, idx
            assert torch.equal(a.cpu(), w), cfg


def test_sharded_keys_every_schedule(tune):
    """pdae_knn_keys_u64 (reference-set sharding): keys carry global indices; slices shorter than k pad with +inf keys."""
    b, r, q, k, world = 1, 4100, 20, 48, 3
    ref = synth.clouds(b, r, seed=9)
    query = ref[:, :q].copy() + np.float32(0.003)
    wd, wi = oracle.knn(ref, query, k)
    R, Q = cu(ref), cu(query)
    cuts = [0, 40, 2500, r]  # the first slice has fewer than k points
    for cfg in SCHEDULES:
        tune(**cfg)
        keys = torch.stack([ops.knn_keys(R[:, cuts[w]:cuts[w + 1]].contiguous(), Q, k, cuts[w]) for w in range(world)])
        D, I = ops.knn_merge_keys(keys)
        assert torch.equal(I.cpu(), torch.from_numpy(wi)), cfg
        assert torch.equal(D.cpu(), torch.from_numpy(wd)), cfg


def test_automatic_plan_on_the_scene_scale_shape_uses_chunks_and_matches_the_oracle(tune):
    """BASELINE config 5 (1 x 100 000 points, 2048 centres, k = 64): chunked + warp-specialised by default."""
    xyz = cu(synth.clouds(1, 100000, seed=11))
    _, center = group.fps(xyz, 2048)
    center = center.contiguous()
    want_nb, want_idx = _oracle_ops.group_points_knn(xyz.cpu(), center.cpu(), 64)
    tune()
    got_nb, got_idx = ops.group_points_knn(xyz, center, 64, want_idx=True)
    assert torch.equal(got_idx.cpu(), want_idx) and torch.equal(got_nb.cpu(), want_nb)
    assert _native.lib().pdae_knn_workspace_bytes(1, 100000, 2048, 3, 64) > 0


@pytest.mark.parametrize("k", [32, 64])
def test_cloud_beyond_one_chunk_without_a_workspace_takes_the_streaming_kernel(tune, k):
    """One chunk numbers its 4-point steps in 16 bits: 4095 tiles of 2048 points (8 386 560 points).  A longer cloud
    without a workspace for chunks is served by the streaming warp-select of knn.cu -- dist / idx, sharded keys,
    Group and raw-gather outputs, all bit for bit the oracle's."""
    r, q = 8_400_000, 16
    assert r > 4095 * 2048 and _native.lib().pdae_knn_workspace_bytes(1, r, q, 3, k) > 0
    tune()
    ref = synth.clouds(1, r, seed=84)
    rng = np.random.default_rng(84)
    query = ref[:, rng.integers(0, r, size=q)] + np.float32(0.001)
    wd, wi = oracle.knn(ref, query, k)
    R, Q = cu(ref), cu(query)
    L, st = _native.lib(), torch.cuda.current_stream().cuda_stream
    dist = torch.empty((1, q, k), dtype=torch.float32, device=DEV)
    idx = torch.empty((1, q, k), dtype=torch.int64, device=DEV)
    assert L.pdae_knn_f32(R.data_ptr(), Q.data_ptr(), 1, r, q, 3, k, 0, dist.data_ptr(), idx.data_ptr(), st) == 0
    assert torch.equal(idx.cpu(), torch.from_numpy(wi)) and torch.equal(dist.cpu(), torch.from_numpy(wd))
    keys = torch.stack([ops.knn_keys(R, Q, k, 0)])
    D, I = ops.knn_merge_keys(keys)
    assert torch.equal(I.cpu(), torch.from_numpy(wi)) and torch.equal(D.cpu(), torch.from_numpy(wd))
    nb = torch.empty((1, q, k, 3), dtype=torch.float32, device=DEV)
    idx.fill_(-1)
    assert L.pdae_group_f32(R.data_ptr(), Q.data_ptr(), 1, r, q, k, idx.data_ptr(), nb.data_ptr(), st) == 0
    assert torch.equal(idx.cpu(), torch.from_numpy(wi))
    assert torch.equal(nb.cpu(), torch.from_numpy(ref[0][wi[0]][None] - query[:, :, None, :]))
    raw, raw_idx = ops.group_points_knn(R, Q, k, want_idx=True, subtract_center=False)  # no workspace on this route
    assert torch.equal(raw_idx.cpu(), torch.from_numpy(wi)) and torch.equal(raw.cpu(), torch.from_numpy(ref[0][wi[0]][None]))
