"""Segment Chamfer (csrc/segchamfer.cu) on packed variable-size clouds, with CUDA events over windows of at least half a
second after warm-up.  Cases (xyz1 and xyz2 drawn with independent seeded segment sizes in the same range):
  equal   128 segments of 2048 against 2048;
  object  128 segments of 512-4096;
  tiny    4096 segments of 16-64;
  scene   8 segments of 40k-120k.
Per case: the segment forward, and forward + L2 loss + backward through SegmentChamferDistanceL2 (atomic and
deterministic gradients).  Next to them the FMA floor sum_s n_s m_s x 6 / 37.2e12 s (six FMA-pipe operations per point
pair at the card's FMA rate, each pair counted once; the segment forward scans every pair in both directions, so its
own floor is twice that).  Comparisons: a Python loop of ops.chamfer_forward over the clouds, ops.segment_knn(1) in
both directions, and on equal segments ops.chamfer_forward(symmetric=False) with the tensor-core filter switched off
(the same scan body, two scans), as it comes (on this shape it takes the tensor-core forward) and the default forward
on the (b, n, 3) view.  The inputs are at most 8 MB and stay in L2, the working set these ops have in
use.  Reads the GPU name, power limit and clock in the same run and writes time_segment_chamfer.json to --out.
usage: python profiles/time_segment_chamfer.py --out DIR"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointdae_b200 import _native, ops, segment_chamfer  # noqa: E402

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


def row(name, ms, floor_ms):
    print("  %-44s %10.3f ms  (floor / time %.1f%%)" % (name, ms, 100 * floor_ms / ms), flush=True)
    return ms


def case(label, s1, s2, seed, equal=False):
    s1, s2 = np.asarray(s1, np.int64), np.asarray(s2, np.int64)
    rng = np.random.default_rng(seed)
    x1 = torch.from_numpy(rng.random((int(s1.sum()), 3), dtype=np.float32)).to(DEV)
    x2 = torch.from_numpy(rng.random((int(s2.sum()), 3), dtype=np.float32)).to(DEV)
    o1 = torch.from_numpy(np.cumsum(s1).astype(np.int32)).to(DEV)
    o2 = torch.from_numpy(np.cumsum(s2).astype(np.int32)).to(DEV)
    pairs = float((s1 * s2).sum())
    floor = pairs * 6 / FMA_RATE * 1e3
    print("%s: %d segments, %d + %d points, floor %.3f ms" % (label, len(s1), int(s1.sum()), int(s2.sum()), floor), flush=True)
    out = {"segments": len(s1), "points1": int(s1.sum()), "points2": int(s2.sum()), "pairs": pairs, "fma_floor_ms": floor}
    out["segment_forward_ms"] = row("segment_chamfer_forward", timed(lambda: ops.segment_chamfer_forward(x1, x2, o1, o2)), floor)
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    loss_fn = segment_chamfer.SegmentChamferDistanceL2()

    def train():
        torch.autograd.grad(loss_fn(a, b, o1, o2), (a, b))

    out["segment_fwd_loss_bwd_ms"] = row("forward + L2 loss + backward", timed(train), floor)
    torch.use_deterministic_algorithms(True)
    out["segment_fwd_loss_bwd_det_ms"] = row("  the same, deterministic", timed(train), floor)
    torch.use_deterministic_algorithms(False)
    starts1, starts2 = np.concatenate(([0], np.cumsum(s1)[:-1])), np.concatenate(([0], np.cumsum(s2)[:-1]))
    views = [(x1[p:p + n].view(1, n, 3), x2[q:q + m].view(1, m, 3)) for p, n, q, m in zip(starts1, s1, starts2, s2)]

    def loop():
        for u, v in views:
            ops.chamfer_forward(u, v)

    out["python_loop_chamfer_forward_ms"] = row("Python loop of ops.chamfer_forward", timed(loop), floor)

    def knn():
        ops.segment_knn(1, x2, x1, o2, o1)
        ops.segment_knn(1, x1, x2, o1, o2)

    out["segment_knn1_both_ms"] = row("segment_knn(1) both directions", timed(knn), floor)
    if equal:
        bsz, n, m = len(s1), int(s1[0]), int(s2[0])
        u, v = x1.view(bsz, n, 3), x2.view(bsz, m, 3)
        lib = _native.lib()
        mode = lib.pdae_tune_chamfer_tc(0, 0.0)  # without the tensor-core filter: the two-scan FP32 form
        try:
            out["chamfer_forward_two_scan_ms"] = row("ops.chamfer_forward(symmetric=False), no TC",
                                                     timed(lambda: ops.chamfer_forward(u, v, symmetric=False)), floor)
        finally:
            lib.pdae_tune_chamfer_tc(mode, 0.0)
        out["chamfer_forward_nosym_tc_ms"] = row("ops.chamfer_forward(symmetric=False)",
                                                 timed(lambda: ops.chamfer_forward(u, v, symmetric=False)), floor)
        out["chamfer_forward_default_ms"] = row("ops.chamfer_forward (default)", timed(lambda: ops.chamfer_forward(u, v)), floor)
        out["segment_over_two_scan"] = out["segment_forward_ms"] / out["chamfer_forward_two_scan_ms"]
        print("  segment / two-scan: %.3f" % out["segment_over_two_scan"], flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    info = gpu_info()
    print(info, flush=True)
    rng = np.random.default_rng(0)
    res = {"gpu": info, "fma_rate_assumed": FMA_RATE,
           "equal_128x2048": case("equal", [2048] * 128, [2048] * 128, 1, equal=True),
           "object_128x512_4096": case("object", rng.integers(512, 4097, 128), rng.integers(512, 4097, 128), 2),
           "tiny_4096x16_64": case("tiny", rng.integers(16, 65, 4096), rng.integers(16, 65, 4096), 3),
           "scene_8x40k_120k": case("scene", rng.integers(40000, 120001, 8), rng.integers(40000, 120001, 8), 4)}
    res["sm_clock_mhz_at_end"] = float(subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader,nounits",
                                                      "-i", "0"], capture_output=True, text=True).stdout.strip())
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "time_segment_chamfer.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
