"""How much of the patchifier branch (FPS -> Group) hides behind the Chamfer branch?  Times graphs of: the loss
branch alone, the patchifier alone, both on two streams (as bench.py does), and both with node priorities."""
import json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from pointdae_b200 import ops, synth, graphs

dev = torch.device("cuda:0")
B, N, G, M, POOL = 128, 2048, 64, 32, 24
base = torch.from_numpy(synth.clouds(B, N, seed=1)).to(dev)
gen = torch.Generator(device="cpu").manual_seed(1)
clouds = [base[torch.randperm(B, generator=gen).to(dev)][:, torch.randperm(N, generator=gen).to(dev)].contiguous() for _ in range(POOL)]
preds = [c + 0.02 * torch.randn_like(c) for c in clouds]
gone = torch.ones(1, device=dev)
side = torch.cuda.Stream()

def loss_branch(i):
    d1, d2, i1, i2 = ops.chamfer_forward(preds[i], clouds[i])
    l = ops.chamfer_mean_loss(d1, d2)
    return ops.chamfer_loss_backward(preds[i], clouds[i], i1, i2, d1, d2, gone, 1.0, 1.0), l

def patch_branch(i):
    _, cen = ops.fps_gather(clouds[i], G)
    return ops.group_points_knn(clouds[i], cen, M, want_idx=False)

def fps_only(i):
    return ops.fps_gather(clouds[i], G)

def both(i):
    main = torch.cuda.current_stream()
    side.wait_stream(main)
    with torch.cuda.stream(side):
        a = patch_branch(i)
    b = loss_branch(i)
    main.wait_stream(side)
    return a, b

def both_serial(i):
    return patch_branch(i), loss_branch(i)

def loss_then_patch(i):
    return loss_branch(i), patch_branch(i)

def time_graphs(fn, prio=None):
    for i in range(3): fn(i)
    torch.cuda.synchronize()
    gs = []
    for i in range(POOL):
        g = graphs.PriorityGraph(low_priority=prio) if prio is not None else torch.cuda.CUDAGraph()
        with (g.capture() if prio is not None else torch.cuda.graph(g)):
            keep = fn(i)
        gs.append((g, keep))
    for g, _ in gs: g.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for r in range(4):
            for g, _ in gs: g.replay()
        b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e3 / (4 * POOL))
    return round(sorted(ts)[2], 2)

out = {
    "loss_branch_us": time_graphs(loss_branch),
    "patch_branch_us": time_graphs(patch_branch),
    "fps_only_us": time_graphs(fps_only),
    "both_two_streams_us": time_graphs(both),
    "both_one_stream_us": time_graphs(both_serial),
    "loss_then_patch_one_stream_us": time_graphs(loss_then_patch),
    "both_prio_patch_low_us": time_graphs(both, prio=("fps_", "knn4_")),
    "both_prio_patch_high_us": time_graphs(both, prio=("chamfer", "fill_keys")),
}
print(json.dumps(out))
