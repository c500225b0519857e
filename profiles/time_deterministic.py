"""Atomic vs deterministic gradients on the GPU: for each gradient both forms are timed in the same call, alternating,
with CUDA events over windows of at least half a second each.  Prints the GPU name and power limit and writes
time_deterministic.json to --out.  usage: python profiles/time_deterministic.py --out DIR"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointdae_b200 import ops, synth  # noqa: E402

DEV = "cuda:0"


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def timed(fn, window=0.5):
    """mean time per call (us) over a window of at least `window` seconds"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    reps = 1
    while True:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        ms = a.elapsed_time(b)
        if ms >= window * 1e3:
            return ms * 1e3 / reps
        reps = max(reps * 2, int(reps * window * 1.2e3 / max(ms, 1e-3)))


def pair(fn, rounds=3):
    """alternate atomic / deterministic; per form the median of the rounds (us)"""
    out = {"atomic": [], "det": []}
    for _ in range(rounds):
        for mode in ("atomic", "det"):
            torch.use_deterministic_algorithms(mode == "det")
            out[mode].append(timed(fn))
    torch.use_deterministic_algorithms(False)
    return {k: float(np.median(v)) for k, v in out.items()} | {"rounds": out}


def chamfer_case(b, n, collapsed=False):
    c = synth.clouds(b, n, seed=1)
    p = synth.prediction(c, seed=1)
    if collapsed:
        p[:] = p[:, :1]
    x1, x2 = cu(p), cu(c)
    d1, d2, i1, i2 = ops.chamfer_forward(x1, x2)
    gone = torch.ones(1, device=DEV)
    return lambda: ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 1.0, 1.0)


def fine_case(b=6528, n=36, m=32):
    rng = np.random.default_rng(0)
    x1, x2 = cu(rng.random((b, n, 3), dtype=np.float32)), cu(rng.random((b, m, 3), dtype=np.float32))
    d1, d2, i1, i2 = ops.chamfer_forward(x1, x2)
    gone = torch.ones(1, device=DEV)
    return lambda: ops.chamfer_loss_backward(x1, x2, i1, i2, d1, d2, gone, 1.0, 1.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    print("gpu:", q)
    rng = np.random.default_rng(1)
    res = {"gpu": q, "unit": "us per call, median of 3 alternating rounds, each a CUDA-event window >= 0.5 s"}
    cases = {
        "chamfer_loss_bwd_128x2048": lambda: chamfer_case(128, 2048),
        "chamfer_loss_bwd_128x2048_collapsed": lambda: chamfer_case(128, 2048, collapsed=True),
        "chamfer_loss_bwd_C2_128x1024": lambda: chamfer_case(128, 1024),
        "chamfer_loss_bwd_fine_6528x36v32": fine_case,
        "chamfer_loss_bwd_C4_256x8192": lambda: chamfer_case(256, 8192),
        "chamfer_loss_bwd_1x100000": lambda: chamfer_case(1, 100000),
    }
    for name, make in cases.items():
        res[name] = pair(make())
        print(name, res[name]["atomic"], res[name]["det"], flush=True)
    # gather grad at C2: 128 clouds of 1024 points, 64 centres, 3 channels
    idx = cu(rng.integers(0, 1024, (128, 64)).astype(np.int32))
    go = torch.randn(128, 3, 64, device=DEV)
    res["gather_grad_C2"] = pair(lambda: ops.gather_points_grad(go, idx, 1024))
    # group_points grad at the 3DETR shape: 16 x 20000 points, 2048 centres x 64, 3 channels
    gi = cu(rng.integers(0, 20000, (16, 2048, 64)).astype(np.int32))
    gg = torch.randn(16, 3, 2048, 64, device=DEV)
    res["group_points_grad_3detr"] = pair(lambda: ops.group_points_grad(gg, gi, 20000))
    # three_interpolate grad: 16 clouds, 4096 -> 1024 points, 128 channels
    ti = cu(rng.integers(0, 1024, (16, 4096, 3)).astype(np.int32))
    tw = torch.rand(16, 4096, 3, device=DEV)
    gt = torch.randn(16, 128, 4096, device=DEV)
    res["three_interpolate_grad_16x4096to1024_c128"] = pair(lambda: ops.three_interpolate_grad(gt, ti, tw, 1024))
    # graph-feature grad at C3 (32 clouds of 1024 points, k = 20)
    for c in (64, 128):
        x = torch.randn(32, c, 1024, device=DEV)
        fidx = ops.feat_knn(x, 20)
        gout = torch.randn(32, 1024, 20, 2 * c, device=DEV)
        res["graph_feature_grad_C3_c%d" % c] = pair(lambda: ops._graph_feature_bwd(gout, fidx, c, 1024))
    for k in ("gather_grad_C2", "group_points_grad_3detr", "three_interpolate_grad_16x4096to1024_c128",
              "graph_feature_grad_C3_c64", "graph_feature_grad_C3_c128"):
        print(k, res[k]["atomic"], res[k]["det"], flush=True)
    # the native step at the headline shape on 4 rotating input sets (128 x 2048 x 3 x 2 x 4 = 25 MB inputs plus the
    # ~270 MB of outputs and workspaces of the 4 buffer sets: larger than the 126 MB L2)
    sets = [(cu(c), cu(synth.prediction(c, seed=s))) for s, c in enumerate(synth.clouds(128, 2048, seed=s + 10) for s in range(4))]
    gone = torch.ones(1, device=DEV)
    for mode in ("atomic", "det"):
        det = mode == "det"
        bufs = [ops.StepBuffers(128, 2048, 128, 32, torch.device(DEV), deterministic=det) for _ in sets]
        state = {"i": 0}

        def step(bufs=bufs, det=det):
            i = state["i"] = (state["i"] + 1) % len(sets)
            ops.hot_step(sets[i][0], sets[i][1], 128, 32, gone, buffers=bufs[i], deterministic=det)
        res.setdefault("step_128x2048", {})[mode] = step
    fa, fd = res["step_128x2048"]["atomic"], res["step_128x2048"]["det"]
    rounds = {"atomic": [], "det": []}
    for _ in range(3):
        rounds["atomic"].append(timed(fa))
        rounds["det"].append(timed(fd))
    res["step_128x2048"] = {k: float(np.median(v)) for k, v in rounds.items()} | {"rounds": rounds}
    print("step_128x2048", res["step_128x2048"]["atomic"], res["step_128x2048"]["det"])
    with open(os.path.join(args.out, "time_deterministic.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
