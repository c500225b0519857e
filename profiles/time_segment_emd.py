"""Segment EMD (csrc/segemd.cu) on packed variable-size clouds, with CUDA events over windows of at least half a second
after warm-up.  Cases (xyz1 and xyz2 drawn with independent seeded segment sizes in the same range):
  equal   128 segments of 2048 against 2048;
  object  128 segments of 512-4096;
  tiny    4096 segments of 16-64;
  large   8 segments of 8192-16384.
Per case: forward (segment_emd_match + segment_emd_cost) and forward + backward (segment_earth_mover_distance and both
gradients).  Next to them the MUFU floor used for the equal-size EMD: 30 pair evaluations per (k,l) in approxmatch, 10
in the cost and 20 in the gradient, one MUFU.EX2 each, at an assumed 16 MUFU results per SM per clock at the card's
maximum SM clock (an assumption, not a measured rate).  Comparison: a Python loop of emd.earth_mover_distance over the
segments (forward, and forward + backward), and on equal segments ops.emd_match + emd_cost (+ emd_cost_grad) on the
(b, n, 3) view.  The inputs are a few MB and stay in L2; the kernels are bound by MUFU.EX2, not by memory.  Reads the
GPU name, power limit and clock in the same run and writes time_segment_emd.json to --out.
usage: python profiles/time_segment_emd.py --out DIR"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointdae_b200 import emd, ops, segment_emd  # noqa: E402

DEV = "cuda:0"
MUFU_PER_SM_CLK = 16


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


def row(name, ms, floor_ms):
    print("  %-46s %10.3f ms  (floor / time %.1f%%)" % (name, ms, 100 * floor_ms / ms), flush=True)
    return ms


def case(label, s1, s2, seed, info, equal=False):
    s1, s2 = np.asarray(s1, np.int64), np.asarray(s2, np.int64)
    rng = np.random.default_rng(seed)
    x1 = torch.from_numpy(rng.standard_normal((int(s1.sum()), 3), dtype=np.float32)).to(DEV)
    x2 = torch.from_numpy(rng.standard_normal((int(s2.sum()), 3), dtype=np.float32)).to(DEV)
    o1 = torch.from_numpy(np.cumsum(s1).astype(np.int32)).to(DEV)
    o2 = torch.from_numpy(np.cumsum(s2).astype(np.int32)).to(DEV)
    pairs = float((s1 * s2).sum())
    rate = MUFU_PER_SM_CLK * info["sms"] * info["max_sm_clock_mhz"] * 1e6
    floor_f, floor_fb = pairs * 40 / rate * 1e3, pairs * 60 / rate * 1e3
    print("%s: %d segments, %d + %d points, MUFU floor fwd %.3f / fwd+bwd %.3f ms" % (
        label, len(s1), int(s1.sum()), int(s2.sum()), floor_f, floor_fb), flush=True)
    out = {"segments": len(s1), "points1": int(s1.sum()), "points2": int(s2.sum()), "pairs": pairs,
           "mufu_floor_fwd_ms": floor_f, "mufu_floor_fwd_bwd_ms": floor_fb}

    def fwd():
        rl, rr = ops.segment_emd_match(x1, x2, o1, o2)
        ops.segment_emd_cost(x1, x2, o1, o2, rl, rr)

    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)

    def fwd_bwd():
        torch.autograd.grad(segment_emd.segment_earth_mover_distance(a, b, o1, o2).sum(), (a, b))

    out["segment_fwd_ms"] = row("segment match + cost", timed(fwd), floor_f)
    out["segment_fwd_bwd_ms"] = row("segment_earth_mover_distance fwd + bwd", timed(fwd_bwd), floor_fb)
    starts1, starts2 = np.concatenate(([0], np.cumsum(s1)[:-1])), np.concatenate(([0], np.cumsum(s2)[:-1]))
    views = [(a[p:p + n].view(1, n, 3), b[q:q + m].view(1, m, 3)) for p, n, q, m in zip(starts1, s1, starts2, s2)]

    def loop_fwd():
        with torch.no_grad():
            for u, v in views:
                emd.earth_mover_distance(u, v)

    def loop_fwd_bwd():
        costs = [emd.earth_mover_distance(u, v) for u, v in views]
        torch.autograd.grad(torch.cat(costs).sum(), (a, b))

    out["python_loop_fwd_ms"] = row("Python loop of emd.earth_mover_distance", timed(loop_fwd), floor_f)
    out["python_loop_fwd_bwd_ms"] = row("  the same, fwd + bwd", timed(loop_fwd_bwd), floor_fb)
    if equal:
        bsz, n, m = len(s1), int(s1[0]), int(s2[0])
        u, v = x1.view(bsz, n, 3), x2.view(bsz, m, 3)
        gc = torch.ones(bsz, device=DEV)

        def eq_fwd():
            rl, rr, _ = ops.emd_match(u, v)
            return rl, rr, ops.emd_cost(u, v, ratio_l=rl, ratio_r=rr)

        def eq_fwd_bwd():
            rl, rr, _ = eq_fwd()
            ops.emd_cost_grad(gc, u, v, ratio_l=rl, ratio_r=rr)

        out["equal_size_fwd_ms"] = row("ops.emd_match + emd_cost on (b, n, 3)", timed(eq_fwd), floor_f)
        out["equal_size_fwd_bwd_ms"] = row("  the same + emd_cost_grad", timed(eq_fwd_bwd), floor_fb)
        out["segment_over_equal_size_fwd"] = out["segment_fwd_ms"] / out["equal_size_fwd_ms"]
        out["segment_over_equal_size_fwd_bwd"] = out["segment_fwd_bwd_ms"] / out["equal_size_fwd_bwd_ms"]
        print("  segment / equal-size: fwd %.3f, fwd + bwd %.3f" % (out["segment_over_equal_size_fwd"],
                                                                   out["segment_over_equal_size_fwd_bwd"]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    info = gpu_info()
    print(info, flush=True)
    rng = np.random.default_rng(0)
    res = {"gpu": info, "mufu_per_sm_clk_assumed": MUFU_PER_SM_CLK,
           "equal_128x2048": case("equal", [2048] * 128, [2048] * 128, 1, info, equal=True),
           "object_128x512_4096": case("object", rng.integers(512, 4097, 128), rng.integers(512, 4097, 128), 2, info),
           "tiny_4096x16_64": case("tiny", rng.integers(16, 65, 4096), rng.integers(16, 65, 4096), 3, info),
           "large_8x8192_16384": case("large", rng.integers(8192, 16385, 8), rng.integers(8192, 16385, 8), 4, info)}
    res["sm_clock_mhz_at_end"] = float(subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits",
                                                      "-i", "0"], capture_output=True, text=True).stdout.strip())
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "time_segment_emd.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
