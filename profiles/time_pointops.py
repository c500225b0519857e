"""Segment FPS and segment kNN (csrc/pointops.cu) on packed variable-size clouds, with CUDA events over windows of at
least half a second after warm-up:
  scene   8 seeded segments of 40k-120k points, FPS to 1/4, kNN 16 of the samples;
  object  128 seeded segments of 512-4096 points, FPS to 1/8, kNN 32 of the samples;
  equal   128 x 2048 in equal segments, FPS to 1/8 and kNN 32, next to ops.fps_gather and ops.knn_points on (128, 2048, 3).
Next to each time: the point pairs the call evaluates (FPS: (samples - 1) x points per segment; kNN: queries x points)
and the FMA floor pairs x 6 / 37.2e12 s (six FMA-pipe operations per pair at the card's FMA rate).  The inputs are a few
MB and stay in L2; that is the working set these ops have in use.  Reads the GPU name, power limit and clock in the
same run and writes time_pointops.json to --out.
usage: python profiles/time_pointops.py --out DIR"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointdae_b200 import ops  # noqa: E402

DEV = "cuda:0"
FMA_RATE = 37.2e12  # FMA-pipe operations per second


def timed(fn, window=0.5):
    """mean time per call (ms) over a window of at least `window` seconds, after 2 warm-up calls"""
    for _ in range(2):
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
            return ms / reps
        reps = max(reps * 2, int(reps * window * 1.2e3 / max(ms, 1e-3)))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "max_sm_clock_mhz": float(q[2]), "sm_clock_mhz_at_start": float(q[3]),
            "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def entry(name, ms, pairs):
    floor = pairs * 6 / FMA_RATE * 1e3
    print("  %-28s %10.3f ms  floor %9.3f ms  (%.1f%%)" % (name, ms, floor, 100 * floor / ms), flush=True)
    return {"ms": ms, "pairs": pairs, "fma_floor_ms": floor, "floor_over_time": floor / ms}


def segment_case(label, sizes, frac, k, seed):
    sizes = np.asarray(sizes, np.int64)
    samples = np.maximum(sizes // frac, 1)
    rng = np.random.default_rng(seed)
    x = torch.from_numpy(rng.random((int(sizes.sum()), 3), dtype=np.float32)).to(DEV)
    off = torch.from_numpy(np.cumsum(sizes).astype(np.int32)).to(DEV)
    noff = torch.from_numpy(np.cumsum(samples).astype(np.int32)).to(DEV)
    n, m = int(sizes.max()), int(samples.sum())
    idx = ops.segment_fps(x, off, noff, n=n, m=m)
    q = x[idx.long()].contiguous()
    print("%s: %d segments, %d points, %d samples" % (label, len(sizes), int(sizes.sum()), m), flush=True)
    out = {"segments": len(sizes), "points": int(sizes.sum()), "largest": n, "samples": m, "k": k,
           "segment_fps": entry("segment_fps", timed(lambda: ops.segment_fps(x, off, noff, n=n, m=m)),
                                float(((samples - 1) * sizes).sum())),
           "segment_knn": entry("segment_knn", timed(lambda: ops.segment_knn(k, x, q, off, noff)),
                                float((samples * sizes).sum()))}
    return out, (x, off, noff, n, m, q)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    info = gpu_info()
    print(info, flush=True)
    rng = np.random.default_rng(0)
    scene, _ = segment_case("scene", rng.integers(40000, 120001, 8), 4, 16, 1)
    obj, _ = segment_case("object", rng.integers(512, 4097, 128), 8, 32, 2)
    equal, (x, off, noff, n, m, q) = segment_case("equal", [2048] * 128, 8, 32, 3)
    xb = x.view(128, 2048, 3)
    qb = q.view(128, 256, 3)
    equal["fps_gather"] = entry("ops.fps_gather (128,2048)->256", timed(lambda: ops.fps_gather(xb, 256)), 255.0 * 2048 * 128)
    equal["knn_points"] = entry("ops.knn_points k=32", timed(lambda: ops.knn_points(xb, qb, 32)), 256.0 * 2048 * 128)
    res = {"gpu": info, "fma_rate_assumed": FMA_RATE, "scene": scene, "object": obj, "equal_128x2048": equal,
           "sm_clock_mhz_at_end": float(subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits",
                                                        "-i", "0"], capture_output=True, text=True).stdout.strip())}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "time_pointops.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
