"""DGCNN feature kNN (16 x 2048 points, k = 20) timing: python profiles/time_featknn.py"""
import json, os, statistics, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointdae_b200 import dgcnn_util, synth
out = {"form": "symmetric"}
for C in (64, 128):
    x = torch.from_numpy(synth.features(16, C, 2048, seed=C)).to("cuda:0")
    for _ in range(3):
        dgcnn_util.knn(x, 20)
    torch.cuda.synchronize()
    ts = []
    for _ in range(7):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); dgcnn_util.knn(x, 20); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    ms = statistics.median(ts)
    out["C=%d" % C] = {"ms": ms, "fma_pipe_frac_C_lane_ops_per_pair": 16 * 2048.0 * 2048 * C / (ms * 1e-3) / (148 * 128 * 1.965e9)}
print(json.dumps(out))
