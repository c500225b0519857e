"""Approximate EMD on the GPU: forward (approxmatch + cost, ratio path) and forward + backward (+ gradient) at
128 x 2048^2 (CTA per cloud), 8 x 2048^2 (clusters) and 256 x 8192^2 (C4), with CUDA events over windows of at least
half a second after warm-up.  Each shape cycles through enough seeded input sets that they exceed the 126 MB L2 or,
when that would take more than 8 sets, through 8 (the inputs are a few MB; the kernels are bound by MUFU.EX2, not by
memory).  Next to each time: the pair evaluations the shape needs (30 per (k,l) in approxmatch, 10 in the cost, 20 in
the gradient) and the floor they imply at 16 MUFU results per SM per clock at the card's maximum SM clock.  Reads the
GPU name, power limit and clock in the same run and writes time_emd.json to --out.
usage: python profiles/time_emd.py --out DIR"""
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
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1]), "max_sm_clock_mhz": float(q[2]),
            "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def case(b, n, info):
    sets = int(min(8, max(2, np.ceil(126e6 / (2 * b * n * 3 * 4)))))
    rng = np.random.default_rng(0)
    data = [(torch.from_numpy(rng.standard_normal((b, n, 3), dtype=np.float32)).to(DEV),
             torch.from_numpy(rng.standard_normal((b, n, 3), dtype=np.float32)).to(DEV)) for _ in range(sets)]
    gc = torch.ones(b, device=DEV)
    it = [0]

    def fwd():
        x1, x2 = data[it[0] % sets]
        it[0] += 1
        rl, rr, _ = ops.emd_match(x1, x2)
        ops.emd_cost(x1, x2, ratio_l=rl, ratio_r=rr)
        return x1, x2, rl, rr

    def fwd_bwd():
        x1, x2, rl, rr = fwd()
        ops.emd_cost_grad(gc, x1, x2, ratio_l=rl, ratio_r=rr)

    def match_only():
        x1, x2 = data[it[0] % sets]
        it[0] += 1
        ops.emd_match(x1, x2)

    pairs = float(b) * n * n
    rate = MUFU_PER_SM_CLK * info["sms"] * info["max_sm_clock_mhz"] * 1e6  # MUFU results per second
    out = {"b": b, "n": n, "m": n, "input_sets": sets}
    for name, fn, evals in (("approxmatch", match_only, 30), ("forward", fwd, 40), ("forward_backward", fwd_bwd, 60)):
        ms = timed(fn)
        floor = evals * pairs / rate * 1e3
        out[name] = {"ms": ms, "pair_evaluations": evals * pairs, "mufu_floor_ms": floor, "floor_over_time": floor / ms,
                     "evaluations_per_s": evals * pairs / (ms * 1e-3)}
        print("%4d x %5d^2 %-16s %9.3f ms  floor %8.3f ms  (%.0f%%)" % (b, n, name, ms, floor, 100 * floor / ms), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    info = gpu_info()
    print(info, flush=True)
    res = {"gpu": info, "mufu_per_sm_per_clock_assumed": MUFU_PER_SM_CLK,
           "cases": [case(128, 2048, info), case(8, 2048, info), case(256, 8192, info)]}
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "time_emd.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
