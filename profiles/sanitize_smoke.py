"""Calls every kernel once on small shapes; run under compute-sanitizer (memcheck / racecheck / initcheck / synccheck)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from pointdae_b200 import ops, synth, group, dgcnn_util, pointnet2_utils, knn_cuda
dev = "cuda:0"
def cu(a): return torch.from_numpy(np.ascontiguousarray(a)).to(dev)
x = cu(synth.adversarial(synth.clouds(3, 700, seed=1), seed=1))
y = cu(synth.clouds(3, 1300, seed=2))
for n in (700, 37, 1300, 2048 + 5):
    pointnet2_utils.furthest_point_sample(cu(synth.clouds(2, n, seed=n)), min(n, 40))
pointnet2_utils.furthest_point_sample(cu(synth.clouds(1, 20000, seed=3)), 16)     # cluster kernel
pointnet2_utils.furthest_point_sample(cu(synth.clouds(1, 200000, seed=4)), 4)     # global fallback
idx, cen = group.fps(x, 33)
ops.group_points_knn(x, cen, 17)
knn_cuda.KNN(5, True)(y, cen)                       # knn4, k<=32
knn_cuda.KNN(40, True)(y, cen)                      # knn4, k<=64
knn_cuda.KNN(100, True)(y, cen)                     # streaming warp-select
knn_cuda.KNN(8, True)(torch.cat([y, y], 2), torch.cat([cen, cen], 2))  # dim 6
big = cu(synth.clouds(1, 9000, seed=5)); knn_cuda.KNN(16, True)(big, big[:, :50].contiguous())  # multi-tile
d = ops.chamfer_forward(x, y); ops.chamfer_forward(x, y, symmetric=False)
ops.chamfer_backward(x, y, d[2], d[3], torch.rand_like(d[0]), torch.rand_like(d[1]))
t = cu(synth.clouds(50, 36, seed=6)); ops.chamfer_forward(t, t[:, :32].contiguous())
k, d2, i2 = ops.chamfer_sharded_local(x, y[:, 100:900].contiguous(), 100); ops.chamfer_unpack_keys(k)
ops.chamfer_min_keys(x, y[:, :0].contiguous(), 0)
for c in (3, 7, 64):
    f = cu(synth.features(2, c, 300, seed=c)).requires_grad_(True)
    g = dgcnn_util.get_graph_feature(f, k=9); g.sum().backward()
bq = pointnet2_utils.ball_query(0.2, 16, y, cen)
gp = pointnet2_utils.grouping_operation(y.transpose(1, 2).contiguous().requires_grad_(True), bq); gp.sum().backward()
go = pointnet2_utils.gather_operation(y.transpose(1, 2).contiguous().requires_grad_(True), idx); go.sum().backward()
# fused loss epilogue + scalar-gradient backward, both recovery kernels, odd query counts (idle warps in knn4)
from pointdae_b200 import _native, chamfer_dist
loss3 = ops.chamfer_mean_loss(d[0], d[1], True)
ops.chamfer_loss_backward(x, y, d[2], d[3], d[0], d[1], torch.ones(1, device=dev), 0.5, 0.5, True)
xp = x.clone().requires_grad_(True); chamfer_dist.ChamferDistanceL2()(xp, y).backward()
tc = _native.lib().pdae_tune_chamfer_tc(0, 0.0)  # FP32-pipe forward; > 128 row groups: warp-per-column recovery
ops.chamfer_forward(cu(synth.clouds(1, 16500, seed=7)), y[:1].contiguous()); _native.lib().pdae_tune_chamfer_tc(tc, 0.0)
q300 = cu(synth.clouds(2, 300, seed=8)); knn_cuda.KNN(20, True)(q300, q300)
# three_nn / three_interpolate
dist3, idx3 = pointnet2_utils.three_nn(y, cen)
w3 = torch.softmax(-dist3, dim=2).contiguous()
feat = torch.rand(3, 7, cen.size(1), device=dev, requires_grad=True)
pointnet2_utils.three_interpolate(feat, idx3, w3).sum().backward()
pointnet2_utils.three_nn(y, cen[:, :2].contiguous())
# column-split Chamfer units (every chunk count, fused and separate row-key unpack), affine corruptions
for nc in (1, 2, 3, 16, 0):
    _native.lib().pdae_tune_chamfer_split(nc); ops.chamfer_forward(y, x); ops.chamfer_forward(x, y, scan_done=torch.cuda.Event())
_native.lib().pdae_tune_chamfer_split(0)
mats = torch.randn(3, 3, 3, 3)
ops.affine_points(x, cen, mats)
ops.group_affine(x, cen, 17, mats, want_idx=True); ops.group_affine(x, cen, 40, mats); ops.group_affine(x, cen, 80, mats[:, :0])
# EdgeConv eval gather (row 4, stage 1): ragged channel / point counts
ops.edge_gather_extremum(torch.randn(2, 70, 300, device=dev), torch.randn(2, 70, 300, device=dev),
                         torch.randint(0, 70, (2, 70, 9), device=dev), torch.randn(300, device=dev), torch.randn(300, device=dev))
torch.cuda.synchronize(); print("sanitize smoke done")
