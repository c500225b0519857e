"""A/B of the 3-D kNN / Group kernels on the BASELINE shapes (run on the B200 box):

    python profiles/tune_knn.py [--out gpurun_out/r02/tune_knn.json] [--quick]

For every shape: the automatic plan (form -1) is the timing baseline and the bit-exact comparator; the kernel is run
over a grid of (form, TMA on/off, chunks along the reference cloud, tile) through pdae_tune_knn, where form is one of the
four (queries per warp, warps per CTA, warp-specialised) shapes the plan chooses from.  Times are CUDA events around
replayed CUDA graphs of `reps` launches on the launching stream.  Prints one JSON object; `fma_frac` = pairs x 6 lane-ops / time / (148 x 128 x sm clock)."""
import argparse
import itertools
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pointdae_b200 import _native, group, ops, synth  # noqa: E402

DEV = "cuda:0"
PEAK = 148 * 128 * 1.965e9  # lane-ops / s


def timed(fn, reps=10, rounds=5):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
        with torch.cuda.graph(g, stream=s):
            for _ in range(reps):
                fn()
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b) / reps)
    return best * 1e3  # us


FORMS = {0: "qw4 nw8 spec", 1: "qw4 nw8", 2: "qw4 nw4", 3: "qw2 nw4"}


def tune(form=-1, tile=-1, nz=-1, tma=-1):
    assert _native.lib().pdae_tune_knn(form, tile, nz, tma) == 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    shapes = [
        # name, b, r, q, k, planar
        ("H group 128x2048 q64 k32", 128, 2048, 64, 32, False),
        ("C2 group 128x1024 q64 k32", 128, 1024, 64, 32, False),
        ("C4 group 256x8192 q512 k32", 256, 8192, 512, 32, False),
        ("C5 group 1x100000 q2048 k64", 1, 100000, 2048, 64, False),
        ("C3 dgcnn layer-1 knn 16x2048 k20 (planar self)", 16, 2048, 2048, 20, True),
    ]
    out = {}
    for name, b, r, q, k, planar in shapes:
        xyz = torch.from_numpy(synth.clouds(b, r, seed=7 + r)).to(DEV)
        if planar:
            x = xyz.transpose(1, 2).contiguous()
            run = lambda: ops.feat_knn(x, k)
        else:
            _, center = group.fps(xyz, q)
            center = center.contiguous()
            run = lambda: ops.group_points_knn(xyz, center, k, want_idx=True)
        pairs = b * q * r
        rec = {"pairs": pairs, "fma_floor_us": pairs * 6 / PEAK * 1e6, "runs": []}
        tune()
        want = run()
        torch.cuda.synchronize()
        ntiles = (r + 2047) // 2048
        grid = [dict(form=-1, tma=-1, nz=-1, tile=-1)]
        if not args.quick:
            nzs = [-1] if ntiles == 1 else sorted({1, 2, 3, 4, 6, 8, 12, 16} & set(range(1, ntiles + 1))) + [-1]
            tiles = (1024, 2048) if ntiles > 1 else (2048,)
            for form, tma, nz, tile in itertools.product(FORMS, (0, 1), nzs, tiles):
                if b * q > 20000 and nz not in (-1, 1):
                    continue
                if form == 0 and ntiles == 1:  # the producer warp only pays off on streamed clouds
                    continue
                grid.append(dict(form=form, tma=tma, nz=nz, tile=tile))
        for cfg in grid:
            tune(**cfg)
            got = run()
            torch.cuda.synchronize()
            same = all((a is None and bb is None) or torch.equal(a, bb) for a, bb in zip(
                got if isinstance(got, tuple) else (got,), want if isinstance(want, tuple) else (want,)))
            t = timed(run)
            rec["runs"].append(dict(cfg, us=t, fma_frac=pairs * 6 / (t * 1e-6) / PEAK, same_as_auto=bool(same)))
        tune()
        best = min(rec["runs"], key=lambda x: x["us"])
        rec["best"] = best
        rec["auto"] = rec["runs"][0]
        print(name, "auto %.1f us | best %.1f us %s (%s)" % (
            rec["auto"]["us"], best["us"], {kk: best[kk] for kk in ("form", "tma", "nz", "tile")},
            FORMS.get(best["form"], "automatic")), flush=True)
        assert all(x["same_as_auto"] for x in rec["runs"]), [x for x in rec["runs"] if not x["same_as_auto"]]
        out[name] = rec
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps({k: {"auto_us": v["auto"]["us"], "best": v["best"]} for k, v in out.items()}))


if __name__ == "__main__":
    main()
