"""bench.py -- clouds/sec of the Point-DAE geometry chain on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic ShapeNet-shaped clouds
(headline shape B=128 clouds per GPU, N=2048 points, G=64 groups, M=32 neighbours):
    FPS(2048->64) + centre gather  ->  kNN(32) + gather + centre-subtract (Group)
    ->  Chamfer L2 forward (prediction vs cloud, 2048 x 2048)  ->  loss = mean + mean
    ->  Chamfer backward (gradient to both clouds through the saved argmin)

Prints ONE JSON line (rank 0).  `value` is device-resident throughput (inputs already in HBM),
`e2e` the same chain through the public module API (Group, ChamferDistanceL2, autograd) with inputs
copied from pinned host memory and the loss read back every step.  `roofline` is the dominant
kernel -- the Chamfer forward, since round 2 the tensor-core filter + exact verification of
csrc/chamfer_tc.cu -- in the survey's unit (algorithmic pairs x 6 FMA-pipe lane-ops against the FP32
FMA-pipe peak) with the FP32-pipe kernels of csrc/chamfer.cu timed beside it; `cpu_baseline` is the
reference's pure-PyTorch CPU path on a bounded sample (oracle/torch_cpu_path.py).
Multi-GPU: batch sharding, one process per GPU, no data-path collective (weak scaling).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B, N, G, M = 128, 2048, 64, 32  # headline shape (per GPU)
POOL = 48                        # distinct resident batches cycled through: 48 * 6.3 MB = 302 MB > 126 MB L2
METRIC = "clouds/sec (FPS+Group+Chamfer fwd/bwd, B=128 N=2048)"
UNIT = "clouds/s"
REF_BUDGET_S = 170.0             # wall-clock budget of the CPU reference arm (it does ~50 clouds/s on 16 cores)


def workload_name():
    return "H: B=%d/GPU, N=%d, FPS->%d centres, kNN %d (Group), ChamferL2 %dx%d fwd+bwd" % (B, N, G, M, N, N)


def config_dict(world):
    """Identical for both arms (the driver compares it): what is computed, never how."""
    return {"workload": workload_name(), "sharding": "batch (no collective)" if world > 1 else "single GPU",
            "l2": "inputs rotate through %d distinct resident batches (%.0f MB > 126 MB L2)" % (POOL, POOL * 2 * B * N * 12 / 1e6)}


# ------------------------------------------------------------------------------------ CPU reference
def run_reference(args):
    """--impl reference: the reference's pure-PyTorch CPU path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import torch_cpu_path as T
    from pointdae_b200 import synth

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # one step = the whole B-cloud batch, like the GPU arm, whenever (warmup + steps) of them fit the time budget (they
    # do for the driver's --steps 20); a longer run times a power-of-two share of the batch per step and says so
    probe_c = torch.from_numpy(synth.clouds(8, N, seed=3))
    probe_p = torch.from_numpy(synth.prediction(probe_c.numpy(), seed=3))
    T.step(probe_c, probe_p, G, M)
    t0 = time.perf_counter()
    T.step(probe_c, probe_p, G, M)
    per_cloud = (time.perf_counter() - t0) / 8
    nc = B
    while nc > 8 and nc * per_cloud * (args.steps + args.warmup) > REF_BUDGET_S:
        nc //= 2
    cloud = torch.from_numpy(synth.clouds(nc, N, seed=1))
    pred = torch.from_numpy(synth.prediction(cloud.numpy(), seed=1))
    for _ in range(args.warmup):
        T.step(cloud, pred, G, M)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        T.step(cloud, pred, G, M)
    dt = time.perf_counter() - t0
    ms = dt / args.steps * 1e3
    value = nc / (dt / args.steps)
    sample = "%d of the %d clouds of a batch per step%s, same N=%d/G=%d/M=%d, pure-PyTorch CPU path (torch FPS loop, " \
             "cdist+topk Group, pairwise ChamferL2 fwd+bwd), %d threads" % (
                 nc, B, "" if nc < B else " (the whole batch)", N, G, M, torch.get_num_threads())
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms * B / nc, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(int(os.environ.get("WORLD_SIZE", "1"))),
        "clouds_per_step": nc,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def cpu_baseline():
    import torch
    from oracle import torch_cpu_path as T
    from pointdae_b200 import synth

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    nc = 16
    cloud = torch.from_numpy(synth.clouds(nc, N, seed=2))
    pred = torch.from_numpy(synth.prediction(cloud.numpy(), seed=2))
    t = T.time_step(cloud, pred, G, M, reps=5, warmup=1)
    return {"value": nc / t, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": "%d of %d clouds, same N=%d/G=%d/M=%d, median of 5 reps, pure-PyTorch CPU path "
                      "(torch FPS loop, cdist+topk Group, pairwise ChamferL2 fwd+bwd)" % (nc, B, N, G, M)}


# ------------------------------------------------------------------- reference CUDA ops, same GPU
def ref_gpu_chain(dev, clouds_d, preds_d, gd1, gd2, our_ms, ours_us=None):
    """Times the REFERENCE's own CUDA ops (rebuilt unmodified for sm_100a into oracle/_ref by oracle/build_ref.py)
    on the same resident inputs, outside the timed region: misc.fps (FPS + transposes + gather, utils/misc.py:13-20),
    a KNN_CUDA-like per-cloud loop for the kNN (KNN_CUDA is not vendored: torch cdist+topk per cloud, the launch
    granularity of its Python loop) + the Group gather (models/PointCAE_transformer.py:76-85), chamfer.forward,
    mean+mean, chamfer.backward.  Evidence for the ">= 3x the reference's kernels" target, not a bench line."""
    import importlib.util
    import torch

    def load(name, rel):
        path = os.path.join(ROOT, "oracle", "_ref", rel)
        if not os.path.exists(path):
            raise RuntimeError("oracle/_ref not built")
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    ext = load("_ext", os.path.join("pointnet2_ext", "_ext.so"))
    cham = load("chamfer", os.path.join("chamfer", "chamfer.so"))

    def parts(i):
        c, p = clouds_d[i % POOL], preds_d[i % POOL]
        t = {}
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        fidx = ext.furthest_point_sampling(c[:, :, :3].contiguous(), G)
        center = ext.gather_points(c.transpose(1, 2).contiguous(), fidx).transpose(1, 2).contiguous()
        ev[1].record()
        idxs = []
        for bi in range(B):  # KNN_CUDA.forward is a Python loop over the batch
            d = torch.cdist(center[bi], c[bi])
            idxs.append(d.topk(M, dim=-1, largest=False)[1])
        idx = torch.stack(idxs, 0) + torch.arange(B, device=dev).view(-1, 1, 1) * N
        nb = c.reshape(B * N, 3)[idx.view(-1)].view(B, G, M, 3) - center.unsqueeze(2)
        ev[2].record()
        d1, d2, i1, i2 = cham.forward(p, c)
        loss = d1.mean() + d2.mean()
        ev[3].record()
        cham.backward(p, c, i1, i2, gd1, gd2)
        ev[4].record()
        torch.cuda.synchronize()
        return [ev[k].elapsed_time(ev[k + 1]) for k in range(4)], float(loss)

    for i in range(3):
        parts(i)
    acc = [[], [], [], []]
    for i in range(10):
        ts, _ = parts(3 + i)
        for k in range(4):
            acc[k].append(ts[k])
    med = [statistics.median(a) for a in acc]
    total = sum(med)
    # SURVEY.md 8f row 1: the scene path's radius grouping at 3DETR scale (one block per cloud in the reference,
    # ball_query_gpu.cu:12-57, a warp per query here), same inputs, same GPU
    ball = None
    try:
        from pointdae_b200 import ops as our_ops, synth as our_synth
        bq_xyz = torch.from_numpy(our_synth.clouds(8, 20000, seed=21)).to(dev)
        bq_new = bq_xyz[:, :2048].contiguous()

        def t_us(fn, reps=5):
            fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                fn()
                b.record()
                torch.cuda.synchronize()
                ts.append(a.elapsed_time(b) * 1e3)
            return statistics.median(ts)

        ref_idx = ext.ball_query(bq_new, bq_xyz, 0.2, 64)
        our_idx = our_ops.ball_query(bq_new, bq_xyz, 0.2, 64)
        g_feat = torch.randn(8, 128, 20000, device=dev)
        ball = {"shape": "8 clouds x 20000 points, 2048 centres, radius 0.2, nsample 64",
                "ball_query_us": {"reference": t_us(lambda: ext.ball_query(bq_new, bq_xyz, 0.2, 64)),
                                  "this_repo": t_us(lambda: our_ops.ball_query(bq_new, bq_xyz, 0.2, 64))},
                "group_points_128ch_us": {"reference": t_us(lambda: ext.group_points(g_feat, ref_idx)),
                                          "this_repo": t_us(lambda: our_ops.group_points(g_feat, our_idx))},
                "same_indices": bool(torch.equal(ref_idx, our_idx))}
        ball["ball_query_speedup"] = ball["ball_query_us"]["reference"] / ball["ball_query_us"]["this_repo"]
        ball["group_points_speedup"] = ball["group_points_128ch_us"]["reference"] / ball["group_points_128ch_us"]["this_repo"]
    except Exception as e:  # evidence only
        ball = {"error": repr(e)[:200]}
    kernels_only = None
    if ours_us:
        # the reference's own compiled kernels only (FPS + gather, chamfer.forward + mean, chamfer.backward) against this
        # repo's kernels for the same three pieces, each timed alone: no stand-in in either term
        mine_ms = (ours_us["fps"] + ours_us["chamfer_fwd"] + ours_us["loss"] + ours_us["chamfer_bwd"]) * 1e-3
        kernels_only = {"reference_ms": med[0] + med[2] + med[3], "this_repo_ms": mine_ms,
                        "speedup": (med[0] + med[2] + med[3]) / mine_ms,
                        "pieces": {"fps+gather": med[0] / (ours_us["fps"] * 1e-3),
                                   "chamfer.forward + mean": med[2] / ((ours_us["chamfer_fwd"] + ours_us["loss"]) * 1e-3),
                                   "chamfer.backward": med[3] / (ours_us["chamfer_bwd"] * 1e-3)}}
    return {"ms_per_step": total, "clouds_per_s": B / (total * 1e-3),
            "ms": {"fps+gather (pointnet2 _ext)": med[0], "knn loop (KNN_CUDA-like torch stand-in) + group": med[1],
                   "chamfer.forward + mean": med[2], "chamfer.backward": med[3]},
            "kernels_only_speedup": kernels_only,
            "ball_query_scene_scale": ball,
            "speedup_of_this_repo_incl_knn_stand_in": total / our_ms,
            "note": "reference CUDA sources compiled unmodified for sm_100a; eager launches, median of 10"}


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = sorted(sm)[len(sm) // 2:]  # upper half = samples under load
        return {"sm_mhz": statistics.median(load), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from pointdae_b200 import chamfer_dist, group, ops, synth
    from pointdae_b200 import graphs as graphs_mod

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the single JSON line
        dist.init_process_group("nccl", device_id=dev)
    if args.patchify == "two":  # the public Group module then also takes the two-launch form (end-to-end arm)
        from pointdae_b200 import _native
        _native.lib().pdae_tune_patchify(0, 1, 8)

    # ---- synthetic inputs: POOL distinct batches resident in HBM (rotated so no step re-reads L2-hot data)
    base_c = synth.clouds(B, N, seed=1000 * 1 + rank)
    base_p = synth.prediction(base_c, seed=rank)
    gen = torch.Generator(device="cpu").manual_seed(20260117 + rank)
    clouds_h = torch.empty((POOL, B, N, 3), dtype=torch.float32).pin_memory()
    preds_h = torch.empty((POOL, B, N, 3), dtype=torch.float32).pin_memory()
    bc, bp = torch.from_numpy(base_c), torch.from_numpy(base_p)
    for i in range(POOL):  # each pool entry: a different permutation of clouds and points + jitter
        pb = torch.randperm(B, generator=gen)
        pn = torch.randperm(N, generator=gen)
        clouds_h[i] = bc[pb][:, pn]
        preds_h[i] = bp[pb][:, pn] + 0.001 * torch.randn((B, N, 3), generator=gen)
    clouds_d = clouds_h.to(dev)
    preds_d = preds_h.to(dev)
    gd1 = torch.full((B, N), 1.0 / (B * N), device=dev)  # d(mean)/d(dist), for the reference-CUDA timing block
    gd2 = torch.full((B, N), 1.0 / (B * N), device=dev)
    gone = torch.ones(1, device=dev)                       # upstream gradient of the scalar loss
    stream = torch.cuda.current_stream()

    side = torch.cuda.Stream(device=dev)
    aux = torch.cuda.Stream(device=dev)

    def patchify(c, overlap_previous=False):
        """FPS + centre gather + kNN + gather + centre-subtract: one launch (csrc/patchify.cu) or the two-launch form"""
        if args.patchify == "fused":
            return ops.fps_group(c, G, M, want_idx=False, overlap_previous=overlap_previous)[2]
        _, center = ops.fps_gather(c, G)
        return ops.group_points_knn(c, center, M, want_idx=False)[0]

    def step_device(i, overlap=True):
        """the chain on resident inputs, straight through the op layer (9 of our kernels: fps, knn3,
        fill_keys, chamfer_min, chamfer_col_recover, loss partial + final, chamfer_bwd own + scatter).  The patchifier
        branch (FPS -> Group) and the loss branch (Chamfer fwd -> loss -> bwd) share no data, so they are
        issued on two streams and overlap on the GPU."""
        c, p = clouds_d[i % POOL], preds_d[i % POOL]
        main = torch.cuda.current_stream()
        br = side if overlap else main
        mode = args.patchifier if overlap else "first"
        if mode == "pdl":
            # the forward, then on the SAME stream the patchifier as a programmatic dependent (it reads only the cloud, the
            # forward triggers its dependents at once: the patchifier's CTAs start as the forward's CTAs exit); loss and
            # backward wait for the forward on the other two streams
            d1, d2, i1, i2 = ops.chamfer_forward(p, c)
            fwd_done = torch.cuda.Event()
            fwd_done.record(main)
            nb = patchify(c, overlap_previous=True)
            aux.wait_event(fwd_done)
            with torch.cuda.stream(aux):
                loss = ops.chamfer_mean_loss(d1, d2)[0]
            side.wait_event(fwd_done)
            with torch.cuda.stream(side):
                gx1, gx2 = ops.chamfer_loss_backward(p, c, i1, i2, d1, d2, gone, 1.0, 1.0)
            main.wait_stream(side)
            main.wait_stream(aux)
            return loss, nb, gx1
        if mode == "overlap" and args.patchify == "fused":  # both branches start together (priorities decide who gets the SMs)
            br.wait_stream(main)
            d1, d2, i1, i2 = ops.chamfer_forward(p, c)
            with torch.cuda.stream(br):
                nb = patchify(c)
        elif mode == "overlap":  # round 1 / FP32-pipe scan: FPS starts with the forward, the kNN fills its wave tail
            br.wait_stream(main)
            with torch.cuda.stream(br):
                _, center = ops.fps_gather(c, G)  # latency-bound, one CTA per cloud: starts at once, costs the scan little
            gate = torch.cuda.Event() if args.knn_gate == "scan" else None
            with ops.chamfer_column_split(False):  # the patchifier branch already fills the scan's wave tail
                d1, d2, i1, i2 = ops.chamfer_forward(p, c, scan_done=gate)
            with torch.cuda.stream(br):
                if gate is not None:
                    br.wait_event(gate)
                nb, _ = ops.group_points_knn(c, center, M, want_idx=False)
        elif mode == "first":  # the model's order: patchify, then (encoder / decoder, not part of this path) the loss
            br = main
            nb = patchify(c)
            d1, d2, i1, i2 = ops.chamfer_forward(p, c)
        elif mode == "split":  # FPS alone first (latency-bound, 18 us), the forward, then the kNN beside loss / backward
            _, center = ops.fps_gather(c, G)
            d1, d2, i1, i2 = ops.chamfer_forward(p, c)
            br.wait_stream(main)
            with torch.cuda.stream(br):
                nb, _ = ops.group_points_knn(c, center, M, want_idx=False)
        elif mode == "tail2":  # the forward, then FPS alone, then the kNN beside loss / backward
            d1, d2, i1, i2 = ops.chamfer_forward(p, c)
            _, center = ops.fps_gather(c, G)
            br.wait_stream(main)
            with torch.cuda.stream(br):
                nb, _ = ops.group_points_knn(c, center, M, want_idx=False)
        else:  # "tail": the forward has the GPU to itself (the tensor-core kernel owns every SM's shared memory and tensor
            # memory, nothing can share an SM with it); the patchifier runs beside the light loss / backward kernels
            d1, d2, i1, i2 = ops.chamfer_forward(p, c)
            br.wait_stream(main)
            with torch.cuda.stream(br):
                nb = patchify(c)
        # the loss value and the gradients are independent consumers of the match (the gradient needs the upstream scalar,
        # not the loss): the reduction runs on a third stream beside the backward kernels
        lst = aux if overlap else main
        lst.wait_stream(main)
        with torch.cuda.stream(lst):
            loss = ops.chamfer_mean_loss(d1, d2)[0]  # mean(dist1) + mean(dist2), fused (2 launches)
        gx1, gx2 = ops.chamfer_loss_backward(p, c, i1, i2, d1, d2, gone, 1.0, 1.0)  # d(loss)/d(points), 2 launches
        main.wait_stream(br)
        main.wait_stream(lst)
        return loss, nb, gx1

    def new_graph():
        return graphs_mod.PriorityGraph() if args.sched == "priority" else torch.cuda.CUDAGraph()

    def capture(g):
        return g.capture() if args.sched == "priority" else torch.cuda.graph(g)

    # one CUDA graph per pool slot: the chain is launch-bound from Python (~30 us of host time per op),
    # so the resident-input measurement replays captured graphs; kernels and arguments are unchanged.
    graphs = []
    step_bufs = [ops.StepBuffers(B, N, G, M, dev) for _ in range(2)] if args.launch == "native" else None
    if args.launch == "native":
        pass  # the step is ONE native call (csrc/step.cu: six launches, a few us of host time): no graph needed
    elif not args.no_graphs:
        for i in range(3):
            step_device(i)
        torch.cuda.synchronize()
        for i in range(POOL):
            g = new_graph()
            with capture(g):
                out = step_device(i)
            graphs.append((g, out))

    def run_step(i):
        """one step of the timed path; returns its outputs (StepBuffers, or the (loss, neighborhood, gpred) tuple)"""
        if step_bufs is not None:
            return ops.hot_step(clouds_d[i % POOL], preds_d[i % POOL], G, M, gone, buffers=step_bufs[i % 2])
        if graphs:
            graphs[i % POOL][0].replay()
            return graphs[i % POOL][1]
        return step_device(i)

    grouper = group.Group(G, M)
    cd_l2 = chamfer_dist.ChamferDistanceL2()
    # end-to-end arm: double-buffered device inputs filled from pinned host memory on a copy stream (the next
    # step's H2D overlaps this step's kernels, as a data loader would), public modules + autograd for the
    # compute, the loss copied back every step and read by the host one step later.
    copy_stream = torch.cuda.Stream(device=dev)
    in_bufs = [(torch.empty((B, N, 3), device=dev), torch.empty((B, N, 3), device=dev)) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_h = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ev = [torch.cuda.Event() for _ in range(2)]

    capturing = [False]

    def pred_source(i):
        """The cloud is the step's host input (the data loader's batch).  The prediction is the decoder's output and
        is born on the device in the model (models/PointCAE_transformer.py:1059-1066), so by default it is taken from
        device memory (a device-to-device copy stands in for the decoder); --e2e-upload both also uploads it."""
        return preds_h[i % POOL] if args.e2e_upload == "both" else preds_d[i % POOL]

    def prefetch(i):
        c_in, p_in = in_bufs[i % 2]
        cur = torch.cuda.current_stream()
        if capturing[0]:
            # inside a graph: fork the copy stream from the capture stream; the join at the end of the graph orders
            # it before the next replay (the other buffer was last read by the previous graph, already complete)
            copy_stream.wait_stream(cur)
            with torch.cuda.stream(copy_stream):
                c_in.detach().copy_(clouds_h[i % POOL], non_blocking=True)
                p_in.detach().copy_(pred_source(i), non_blocking=True)
            return
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[i % 2])
            c_in.detach().copy_(clouds_h[i % POOL], non_blocking=True)
            p_in.detach().copy_(pred_source(i), non_blocking=True)
            ready[i % 2].record(copy_stream)

    def e2e_body(i):
        """what one end-to-end step enqueues: prefetch of the NEXT batch (pinned host -> device, copy stream),
        the public modules + autograd on THIS batch, the loss copied to pinned host memory."""
        prefetch(i + 1)
        c_in, p_in = in_bufs[i % 2]
        if args.patchifier == "first":
            nb, center = grouper(c_in)
            loss = cd_l2(p_in, c_in)
            side.wait_stream(torch.cuda.current_stream())  # (keeps the join below valid inside a capture)
        elif args.patchifier in ("tail", "pdl", "split", "tail2"):  # (the Group module runs FPS and kNN back to back: no split here)
            loss = cd_l2(p_in, c_in)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                nb, center = grouper(c_in)
        elif args.knn_gate == "scan":
            side.wait_stream(torch.cuda.current_stream())
            gate = torch.cuda.Event()
            with ops.chamfer_scan_event(gate):  # recorded between the Chamfer scan and its column recovery
                loss = cd_l2(p_in, c_in)
            with torch.cuda.stream(side):
                nb, center = grouper(c_in, knn_after=gate)  # FPS at once, kNN once the scan is done
        else:
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                nb, center = grouper(c_in)
            with ops.chamfer_column_split(False):  # the patchifier on `side` already fills the scan's wave tail
                loss = cd_l2(p_in, c_in)
        loss.backward()
        torch.cuda.current_stream().wait_stream(side)
        loss_h[i % 2].copy_(loss.detach(), non_blocking=True)
        return nb, center

    for c_in, p_in in in_bufs:
        p_in.requires_grad_(True)

    e2e_graphs = []

    def step_e2e(i, first):
        """one end-to-end step; returns the loss of the previous step (read by the host one step late)."""
        cur = torch.cuda.current_stream()
        if first:
            for ev in consumed:
                ev.record(cur)
            prefetch(i)
            cur.wait_event(ready[i % 2])
        if e2e_graphs:
            e2e_graphs[i % POOL][0].replay()
        else:
            cur.wait_event(ready[i % 2])
            in_bufs[i % 2][1].grad = None
            e2e_body(i)
            consumed[i % 2].record(cur)
        loss_ev[i % 2].record(cur)
        if not first:
            loss_ev[(i - 1) % 2].synchronize()
            return float(loss_h[(i - 1) % 2])
        return None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident timing ----------------------------------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # at least 100 untimed steps (~15 ms) right before the timed ones, so clocks are at their loaded state when timing starts
    for i in range(max(args.warmup, 100)):
        run_step(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # exactly --steps timed steps; ms_per_step is their mean
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        outputs = run_step(args.warmup + i)
    e1.record(stream)
    barrier()
    if args.dump_outputs and rank == 0:  # before any later call reuses the step's buffers
        dump_outputs(args.dump_outputs, outputs)
    total_ms = max_over_ranks(e0.elapsed_time(e1))
    ms_per_step = total_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)
    # dominant kernel, timed live with CUDA events on its launching stream: the Chamfer forward alone (no co-running
    # branch), once per timed step over the same rotating pool.  Launched from Python each forward is three kernels
    # with ~10 us of host gaps between them, so the launches are captured 8 forwards per graph and the event pair
    # brackets the replays (events cannot be read out of a replayed graph): ms_per_launch = elapsed / forwards.
    FW = 8
    n_fwd = max(FW, (args.steps // FW) * FW)

    def time_forward(split):
        """split=True: the library's default for a forward that has the GPU to itself (512-row blocks cut into column
        chunks when that evens out the SMs); False: one CTA per row block, the form the overlapped step uses."""
        fwd_graphs = []
        with ops.chamfer_column_split(split):
            if not args.no_graphs:
                for g0 in range(0, POOL, FW):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        keep = [ops.chamfer_forward(preds_d[(g0 + j) % POOL], clouds_d[(g0 + j) % POOL]) for j in range(FW)]
                    fwd_graphs.append((g, keep))
            for r in range(2):  # second pass is the timed one
                e0.record(stream)
                for i in range(n_fwd // FW):
                    if fwd_graphs:
                        fwd_graphs[i % len(fwd_graphs)][0].replay()
                    else:
                        for j in range(FW):
                            ops.chamfer_forward(preds_d[(i * FW + j) % POOL], clouds_d[(i * FW + j) % POOL])
                e1.record(stream)
                torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n_fwd

    from pointdae_b200 import _native as _nat
    tc_mode = _nat.lib().pdae_tune_chamfer_tc(-1, 0.0)  # 0: FP32-pipe kernels only; 1-3: tensor-core filter (default 3)
    cham_ms = time_forward(True)                        # the forward as the timed step launches it (library default)
    _nat.lib().pdae_tune_chamfer_tc(0, 0.0)
    cham_fp32_unsplit_ms = time_forward(False)          # FP32-pipe symmetric kernel, one CTA per 512-row block (round 1)
    cham_fp32_ms = time_forward(True)                   # ... with column-split units
    _nat.lib().pdae_tune_chamfer_tc(tc_mode, 0.0)
    if tc_mode == 0:
        cham_ms = cham_fp32_unsplit_ms

    # ---- end-to-end timing (host buffers, public API) -----------------------------------------------
    for i in range(3):  # eager warm-up (also what --no-graphs measures)
        step_e2e(i, first=(i == 0))
    torch.cuda.synchronize()
    if not args.no_graphs:
        # one CUDA graph per pool slot holding exactly what e2e_body enqueues (H2D of the next batch from pinned
        # memory, Group, ChamferDistanceL2 forward, autograd backward, D2H of the loss)
        capturing[0] = True
        for i in range(POOL):
            in_bufs[i % 2][1].grad = None
            g = new_graph()
            with capture(g):
                keep = e2e_body(i)
                torch.cuda.current_stream().wait_stream(copy_stream)
            e2e_graphs.append((g, keep, in_bufs[i % 2][1].grad))
        capturing[0] = False
    for i in range(max(args.warmup, 100)):
        step_e2e(i, first=(i == 0))
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    e2e_first = max(args.warmup, 100)
    e2e_steps = args.steps
    for i in range(e2e_steps):  # the warm-up left the next batch prefetched: the timed steps continue its pipeline
        step_e2e(e2e_first + i, first=False)
    e1.record(stream)
    barrier()
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)) / e2e_steps
    # sanity (outside the timed region): the loss the e2e arm read back for its last step equals the loss of the
    # device-resident chain on the same pool slot
    last = e2e_first + e2e_steps - 1
    loss_ev[last % 2].synchronize()
    e2e_loss = float(loss_h[last % 2])
    dev_loss = float(step_device(last, overlap=False)[0])
    e2e_checked = abs(e2e_loss - dev_loss) <= 1e-6 * abs(dev_loss)
    if not e2e_checked:
        raise RuntimeError("e2e loss %.9g != device-chain loss %.9g" % (e2e_loss, dev_loss))
    # ---- end to end through the native step call (ops.hot_step = pdae_step_f32): the same double-buffered inputs, the
    # next batch copied from pinned host memory on the copy stream, the loss copied back and read one step late
    e2e_native_ms = None
    if step_bufs is not None:
        e2e_bufs = [ops.StepBuffers(B, N, G, M, dev) for _ in range(2)]
        readback = torch.cuda.Stream(device=dev)

        def step_e2e_native(i, first):
            cur = torch.cuda.current_stream()
            if first:
                for ev in consumed:
                    ev.record(cur)
                prefetch(i)
            cur.wait_event(ready[i % 2])
            prefetch(i + 1)
            c_in, p_in = in_bufs[i % 2]
            o = ops.hot_step(c_in.detach(), p_in.detach(), G, M, gone, buffers=e2e_bufs[i % 2])
            consumed[i % 2].record(cur)
            # the 4-byte read-back rides on its own stream: the next step's forward does not queue behind the copy engine
            readback.wait_event(consumed[i % 2])
            with torch.cuda.stream(readback):
                loss_h[i % 2].copy_(o.loss3[0], non_blocking=True)
                loss_ev[i % 2].record(readback)
            if not first:
                loss_ev[(i - 1) % 2].synchronize()
                return float(loss_h[(i - 1) % 2])
            return None

        torch.cuda.synchronize()
        for i in range(max(args.warmup, 100)):
            step_e2e_native(i, first=(i == 0))
        barrier()
        t0 = time.perf_counter()
        e0.record(stream)
        for i in range(e2e_steps):
            step_e2e_native(e2e_first + i, first=False)
        e1.record(stream)
        barrier()
        e2e_native_ms = max_over_ranks(max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)) / e2e_steps
        loss_ev[last % 2].synchronize()
        nat_e2e_loss = float(loss_h[last % 2])
        if abs(nat_e2e_loss - dev_loss) > 1e-6 * abs(dev_loss):
            raise RuntimeError("native e2e loss %.9g != device-chain loss %.9g" % (nat_e2e_loss, dev_loss))
    if step_bufs is not None:  # ... and so does the native step call the resident arm timed
        nat_loss = float(ops.hot_step(clouds_d[last % POOL], preds_d[last % POOL], G, M, gone, buffers=step_bufs[0]).loss3[0])
        if abs(nat_loss - dev_loss) > 1e-6 * abs(dev_loss):
            raise RuntimeError("native step loss %.9g != device-chain loss %.9g" % (nat_loss, dev_loss))
    clocks = sampler.stop() if rank == 0 else None
    # PCIe floor: the step's host -> device copy alone, every rank at once
    barrier()
    e0.record(stream)
    for i in range(50):
        in_bufs[i % 2][0].detach().copy_(clouds_h[i % POOL], non_blocking=True)
        if args.e2e_upload == "both":
            in_bufs[i % 2][1].detach().copy_(preds_h[i % POOL], non_blocking=True)
    e1.record(stream)
    barrier()
    h2d_only_ms = max_over_ranks(e0.elapsed_time(e1)) / 50
    peaks_all = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks_all = json.load(f)
    except Exception:
        pass
    configs = None
    sharded_c5 = None
    if not args.no_configs:
        try:
            configs = config_blocks(dev, peaks_all, world, max_over_ranks)
        except Exception as e:  # evidence only
            configs = {"error": repr(e)[:300]}
        if world > 1:
            try:
                sharded_c5 = sharded_c5_block(dev, world, rank, max_over_ranks)
            except Exception as e:
                sharded_c5 = {"error": repr(e)[:300]}

    if rank == 0:
        props = torch.cuda.get_device_properties(local)
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        sm_max_mhz = float(peaks.get("sm_max_mhz", 1965.0))
        peak_tflops = props.multi_processor_count * 128 * 2 * sm_max_mhz * 1e6 / 1e12  # FP32 FMA pipe, FMA = 2
        pairs = 2.0 * B * N * N  # algorithmic: every (query, reference) pair of both directions
        # 6 FMA-pipe lane-ops per point pair (3 FADD, 1 FMUL, 2 FFMA), each counted as one FMA slot = 2 FLOP
        achieved = pairs * 6 * 2 / (cham_ms * 1e-3) / 1e12                     # the form inside the timed step
        ach_fp32_unsplit = pairs * 6 * 2 / (cham_fp32_unsplit_ms * 1e-3) / 1e12
        ach_fp32 = pairs * 6 * 2 / (cham_fp32_ms * 1e-3) / 1e12
        fp32_forms = {
            "one_cta_per_row_block": {"ms_per_launch": cham_fp32_unsplit_ms, "frac": ach_fp32_unsplit / peak_tflops,
                                      "executed_frac": 0.5 * ach_fp32_unsplit / peak_tflops},
            "column_split_units": {"ms_per_launch": cham_fp32_ms, "frac": ach_fp32 / peak_tflops,
                                   "executed_frac": 0.5 * ach_fp32 / peak_tflops},
            "note": "fill_keys + chamfer_min_kernel<4,128,1,SYM> + chamfer_col_recover_list_kernel (csrc/chamfer.cu): every "
                    "unordered pair evaluated once on the FP32 FMA pipe for both directions, so the pipe executes half the "
                    "algorithmic count (executed_frac); still the path of clouds outside 512..2048 points and of the "
                    "sharded entry points",
        }
        if tc_mode > 0:
            ntile = 2 * B * (N // 128) * (N // 256)  # 128-row x 256-column accumulator tiles of one forward
            mmas = 1 if tc_mode == 3 else 2
            tensor_tflops = ntile * mmas * 2.0 * 128 * 256 * (16 if tc_mode == 3 else 8) / (cham_ms * 1e-3) / 1e12
            roofline = {
                "kernel": "Chamfer forward as the timed step launches it = chamfer_tc_kernel<256,%s> (csrc/chamfer_tc.cu): "
                          "tcgen05 %s products of hi/lo split coordinates into tensor memory, 32-column group minima + "
                          "candidate lists in the epilogue warps, exact FP32 re-evaluation of the surviving groups (bit-"
                          "identical results); one launch" % ("fp16" if tc_mode == 3 else "tf32",
                                                            "kind::f16" if tc_mode == 3 else "kind::tf32"),
                "bound": "fp32-fma-pipe (the survey's unit for this op; the kernel itself is bound by the ALU pipe's FMNMX3 "
                         "rate and by tensor-memory capacity x MMA latency, see tensor_filter)",
                "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s", "frac": achieved / peak_tflops,
                "traffic": 6.35e6,
                "traffic_source": "constant: dram__bytes_read.sum + dram__bytes_write.sum of one launch in profiles/r02/"
                                  "ncu_chamfer_tc_summary.csv (ncu --set full: 6.35 MB read = both clouds once, 0 written -- the 4 MB "
                                  "of results are still in L2 when the kernel ends); not re-measured in this run",
                "note": "achieved = ALGORITHMIC 2*B*N*N pairs x 6 FMA-pipe lane-ops x 2 / CUDA-event time per forward "
                        "(launched alone, 8 forwards per replayed graph); peak = SMs x 128 lanes x 2 x sm_max_mhz (%s). frac "
                        "> 1: the pair distances are evaluated on the tensor cores (approximately) and only ~1.03 groups of "
                        "32 columns per row are evaluated exactly on the FP32 pipe, so the FP32 pipe executes ~1.6 %% of the "
                        "algorithmic count. Algorithmic bytes 10.5 MB (2 clouds in, 4 arrays out) -- not HBM-bound" % (
                            "MEASURED_PEAKS.json" if peaks else "fallback 1965 MHz"),
                "ms_per_launch": cham_ms,
                "share_of_step": cham_ms / ms_per_step,
                "tensor_filter": {
                    "tiles_128x256": ntile, "mma_per_tile": mmas, "tensor_tflops_executed": tensor_tflops,
                    "cycles_per_tile_per_sm": cham_ms * 1e-3 * sm_max_mhz * 1e6 / (ntile / props.multi_processor_count),
                    "ncu": "profiles/r02/ncu_chamfer_tc_summary.csv: ALU pipe ~50 %% active (18 FMNMX3 per 32 values at "
                           "half rate are the floor: ~290 of the ~690 cycles a tile takes on a scheduler), tensor pipe ~25 %%, "
                           "issue ~45 %%",
                    "pipeline": "profiles/r02/trace_chamfer_tc.txt: accumulator free -> MMAs committed -> ready -> read "
                                "-> released, per tile (clock64 stamps)"},
                "fp32_pipe_forms": fp32_forms,
            }
        else:
            roofline = {
                "kernel": "Chamfer forward (PDAE_CHAMFER_TC=0) = fill_keys + chamfer_min_kernel<4,128,1,SYM> + "
                          "chamfer_col_recover_list_kernel",
                "bound": "fp32-fma-pipe", "achieved": achieved, "peak": peak_tflops, "unit": "TFLOP/s",
                "frac": achieved / peak_tflops, "traffic": 8.44e6,
                "traffic_source": "constant: profiles/r01/ncu_full_chamfer_symmetric_summary.csv",
                "executed_frac": 0.5 * achieved / peak_tflops, "ms_per_launch": cham_ms,
                "share_of_step": cham_ms / ms_per_step, "fp32_pipe_forms": fp32_forms,
            }
        # patchifier (1 fused launch, or fps + knn), chamfer forward (1 or 3), loss x2, backward x2
        fused_patchifier = args.patchify == "fused" and args.patchifier in ("tail", "pdl", "first", "overlap")
        launches_per_step = (7 if tc_mode > 0 else 9) - (1 if fused_patchifier else 0)
        try:
            others = other_kernels(dev, clouds_d, preds_d, peaks, props) if world == 1 else None
        except Exception as e:  # evidence only
            others = {"error": repr(e)[:200]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": config_dict(world),
            "launch": "one native call per step (pdae_step_f32, csrc/step.cu: six launches issued from C++ on the caller's stream + "
                      "two library-owned streams): Chamfer forward -> (FPS+Group as a programmatic dependent launch || loss || "
                      "backward)" if args.launch == "native" else ("eager, 3 streams" if args.no_graphs else "CUDA graph per pool slot, 3 streams") + {
                "tail": ": Chamfer forward -> (FPS+Group || loss || backward)",
                "pdl": ": Chamfer forward -> (FPS+Group as a programmatic dependent launch || loss || backward)",
                "split": ": FPS -> Chamfer forward -> (Group || loss || backward)",
                "tail2": ": Chamfer forward -> FPS -> (Group || loss || backward)",
                "first": ": FPS+Group -> Chamfer forward -> (loss || backward)",
                "overlap": ": FPS+Group || Chamfer forward -> (loss || backward)"}[args.patchifier] + (
                "; kNN gated behind the Chamfer scan" if args.knn_gate == "scan" else "") + (
                "; FPS+Group = one launch (FPS warps + kNN consumer warps per cloud)" if fused_patchifier else ""),
            "timed_steps": args.steps, "timed_region_ms": total_ms,
            "e2e": {"value": world * B / ((e2e_native_ms or e2e_ms) * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": (2 if args.e2e_upload == "both" else 1) * B * N * 12,
                    "h2d_only_ms_per_step": h2d_only_ms,
                    "h2d_note": "h2d_only_ms_per_step = the same pinned-host -> device copy alone, all ranks at once (max "
                                "over ranks): the PCIe floor of the step on this box; uploads: %s" % (
                                    "cloud + prediction" if args.e2e_upload == "both" else
                                    "the cloud (the prediction is a device-side product of the model)"),
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_native_ms or e2e_ms, "loss_checked_against_device_chain": e2e_checked,
                    "modules": {"value": world * B / (e2e_ms * 1e-3), "ms_per_step": e2e_ms,
                                "how": "the same step through the reference-facing modules (Group, ChamferDistanceL2, autograd)"
                                       + ("" if args.no_graphs else ", replayed as a CUDA graph")},
                    "how": ("one ops.hot_step call per step (pdae_step_f32: forward, patchifier, loss, gradients) on "
                            "double-buffered inputs; every step copies the next batch from pinned host memory on a copy stream "
                            "and the loss back to the host, read one step late (a training step: patches and gradients stay on "
                            "the device); `modules` = " if e2e_native_ms else "") +
                           "public modules (Group, ChamferDistanceL2, autograd) on double-buffered inputs; every step "
                           "copies the next batch from pinned host memory and the loss back to the host (a training step: "
                           "patches and gradients stay on the device)" + (
                               "" if args.no_graphs else "; the step is replayed as a CUDA graph")},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline,
            "other_kernels": others,
            "configs": configs,
            "sharded_c5": sharded_c5,
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        if world == 1 and not args.no_ref_gpu:
            try:
                ours_us = None
                if isinstance(others, dict) and "error" not in others:
                    ours_us = {"fps": others["fps+centre gather %dx%d->%d" % (B, N, G)]["us"], "chamfer_fwd": cham_ms * 1e3,
                               "loss": others["chamfer mean loss (2 launches)"]["us"],
                               "chamfer_bwd": others["chamfer backward (2 launches)"]["us"]}
                line["ref_gpu"] = ref_gpu_chain(dev, clouds_d, preds_d, gd1, gd2, ms_per_step, ours_us)
            except Exception as e:  # evidence only; never part of the measured arm
                line["ref_gpu"] = {"unavailable": str(e)[:200]}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def _median_ms(fn, reps=5, warm=2):
    """median device time of one call.  Calls shorter than ~0.3 ms are launch-bound from Python (20-30 us of host time per
    op), so they are replayed eight at a time from a CUDA graph (same kernels, same arguments) and the time is divided."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()

    def timed(run, per):
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / per)
        return statistics.median(ts)

    t = timed(fn, 1)
    if t < 0.3:
        try:
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                keep = [fn() for _ in range(8)]
            g.replay()
            torch.cuda.synchronize()
            t = min(t, timed(g.replay, 8))
            del keep
        except Exception:
            torch.cuda.synchronize()
    return t


def config_blocks(dev, peaks, world, max_over_ranks):
    """BASELINE.json configs 2-5 at their full per-GPU size, every kernel of the path timed alone on the device (median of
    5, CUDA events; outside the timed region) with its roofline fraction.  Under torchrun every rank runs its own share
    (C3 is "batch-sharded over 8 B200": B=128 -> 128/world clouds per rank; C2/C4 keep the per-GPU batch; C5 here is
    the unsharded single-GPU form, the sharded form is the `sharded_c5` block) and the times are the max over ranks."""
    import torch
    from pointdae_b200 import dgcnn_util, ops, synth

    fma = 148 * 128 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6  # lane-ops / s
    hbm = float(peaks.get("hbm_gbs", 6556.5))

    def cloud(b, n, seed):
        base = torch.from_numpy(synth.clouds(min(b, 8), n, seed=seed)).to(dev)
        return (base.repeat((b + base.size(0) - 1) // base.size(0), 1, 1)[:b].contiguous()
                + 0.001 * torch.randn(b, n, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(seed)))

    def entry(ms, pairs=None, nbytes=None, **kw):
        ms = max_over_ranks(ms)
        e = {"ms": ms}
        if pairs is not None:
            e["fma_pipe_frac_algorithmic"] = pairs * 6.0 / (ms * 1e-3) / fma
        if nbytes is not None:
            e["GBps"] = nbytes / (ms * 1e-3) / 1e9
            e["hbm_frac"] = e["GBps"] / hbm
        e.update(kw)
        return e

    out = {"peaks": {"fma_lane_ops_per_s": fma, "hbm_GBps": hbm, "source": "MEASURED_PEAKS.json" if peaks else "fallback"}}
    # ---- C2: transformer pretrain, B=128, N=1024, 64 x 32 groups, ChamferL2 (coarse 64^2 and ~5000 fine clouds of 36 x 32)
    c = cloud(128, 1024, 2)
    cen = ops.fps_gather(c, 64)[1]
    fa, fb = cloud(5000, 36, 3), cloud(5000, 32, 4)
    p = c + 0.01 * torch.randn_like(c)
    out["C2 B=128 N=1024 G=64 M=32"] = {
        "fps 1024->64": entry(_median_ms(lambda: ops.fps_gather(c, 64)), us_per_iteration_note="63 sequential iterations"),
        "group k=32": entry(_median_ms(lambda: ops.group_points_knn(c, cen, 32, want_idx=False)), pairs=128 * 64 * 1024),
        "chamfer fwd 128x1024^2": entry(_median_ms(lambda: ops.chamfer_forward(p, c)), pairs=2.0 * 128 * 1024 * 1024),
        "chamfer fwd fine 5000x36x32": entry(_median_ms(lambda: ops.chamfer_forward(fa, fb)), pairs=2.0 * 5000 * 36 * 32),
        "patchifier, one launch (fps + group k=32)": entry(_median_ms(lambda: ops.fps_group(c, 64, 32))),
    }
    # the whole C2 step (patchifier + coarse ChamferL2 forward + loss + backward) as the native call, 200 steps back to back
    gone = torch.ones(1, device=dev)
    bufs = ops.StepBuffers(128, 1024, 64, 32, dev)
    for _ in range(20):
        ops.hot_step(c, p, 64, 32, gone, buffers=bufs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(200):
        ops.hot_step(c, p, 64, 32, gone, buffers=bufs)
    e1.record()
    torch.cuda.synchronize()
    step_ms = max_over_ranks(e0.elapsed_time(e1) / 200)
    out["C2 B=128 N=1024 G=64 M=32"]["step (pdae_step_f32: patchifier + ChamferL2 fwd + loss + bwd)"] = {
        "ms": step_ms, "clouds_per_s_per_gpu": 128 / (step_ms * 1e-3)}
    del c, cen, fa, fb, p, bufs
    # ---- C3: DGCNN k=20 at N=2048, batch-sharded: 128 clouds / world per rank (16 per GPU on 8)
    b3 = 16  # the per-GPU share of the 8-GPU configuration, whatever the world size of this run
    c3 = {"clouds_per_rank": b3, "note": "feature kNN: algorithmic work = C FMA-pipe lane-ops per point pair (the "
                                         "reference's expanded-form GEMM); C=3 runs the 3-D kernel (6 lane-ops per pair)"}
    for C in (3, 64, 128):
        x = torch.from_numpy(synth.features(b3, C, 2048, seed=C)).to(dev)
        idx = dgcnn_util.knn(x, 20)
        ms = max_over_ranks(_median_ms(lambda: dgcnn_util.knn(x, 20), reps=3))
        c3["knn C=%d" % C] = {"ms": ms, "fma_pipe_frac": b3 * 2048.0 * 2048 * (6.0 if C == 3 else C) / (ms * 1e-3) / fma}
        nbytes = b3 * 2048 * 20 * 2 * C * 4 + b3 * C * 2048 * 4 + b3 * 2048 * 20 * 8
        c3["graph feature C=%d" % C] = entry(_median_ms(lambda: ops._graph_feature_fwd(x, idx), reps=3), nbytes=nbytes)
        del x, idx
    # the EdgeConv layers that consume the graph feature (SURVEY.md 8f row 4): tensor-core route against the reference's own
    # layer sequence (get_graph_feature -> Conv2d -> BatchNorm2d -> LeakyReLU -> max, models/dgcnn_util.py:114-128) run by
    # torch on the same GPU with its defaults, training mode, forward + backward
    import torch.nn as nn

    def ref_layer(x, idx, block):
        bb, cc, nn_ = x.shape
        kk = idx.size(2)
        flat = (idx + torch.arange(bb, device=x.device).view(-1, 1, 1) * nn_).view(-1)
        xt = x.transpose(2, 1).contiguous()
        neigh = xt.view(bb * nn_, cc)[flat, :].view(bb, nn_, kk, cc)
        xi = xt.view(bb, nn_, 1, cc).repeat(1, 1, kk, 1)
        return block(torch.cat((neigh - xi, xi), dim=3).permute(0, 3, 1, 2).contiguous()).max(dim=-1, keepdim=False)[0]

    for C, Co in ((3, 64), (64, 64), (64, 128), (128, 256)):
        x = torch.from_numpy(synth.features(b3, C, 2048, seed=C + Co)).to(dev)
        idx = dgcnn_util.knn(x, 20)
        block = nn.Sequential(nn.Conv2d(2 * C, Co, 1, bias=False), nn.BatchNorm2d(Co), nn.LeakyReLU(0.2)).to(dev).train()
        up = torch.randn(b3, Co, 2048, device=dev)

        def step(fn):
            xx = x.clone().requires_grad_(True)
            (fn(xx) * up).sum().backward()

        mine = max_over_ranks(_median_ms(lambda: step(lambda xx: ops.edge_conv(xx, idx, block[0].weight, block[1], 0.2)), reps=3))
        ref = max_over_ranks(_median_ms(lambda: step(lambda xx: ref_layer(xx, idx, block)), reps=3))
        c3["edgeconv %d->%d fwd+bwd (train)" % (C, Co)] = {"ms": mine, "reference_torch_sequence_ms": ref, "speedup": ref / mine}
        del x, idx, block, up
    a1, a2 = cloud(b3, 1024, 7), cloud(b3, 1024, 8)
    c3["chamferL1 fwd %dx1024^2" % b3] = entry(_median_ms(lambda: ops.chamfer_forward(a1, a2)), pairs=2.0 * b3 * 1024 * 1024)
    out["C3 DGCNN k=20 N=2048 (batch-sharded)"] = c3
    del a1, a2
    # ---- C4: B=256, N=8192 -> FPS 512, kNN 32, ChamferL2 8192^2
    c = cloud(256, 8192, 5)
    cen = ops.fps_gather(c, 512)[1]
    p = c + 0.01 * torch.randn_like(c)
    d1, d2, i1, i2 = ops.chamfer_forward(p, c)
    g = torch.full_like(d1, 1e-6)
    out["C4 B=256 N=8192 G=512 M=32"] = {
        "fps 8192->512": entry(_median_ms(lambda: ops.fps_gather(c, 512), reps=3)),
        "group k=32": entry(_median_ms(lambda: ops.group_points_knn(c, cen, 32, want_idx=False), reps=3), pairs=256.0 * 512 * 8192),
        "chamfer fwd 256x8192^2": entry(_median_ms(lambda: ops.chamfer_forward(p, c), reps=3), pairs=2.0 * 256 * 8192 * 8192),
        "chamfer bwd": entry(_median_ms(lambda: ops.chamfer_backward(p, c, i1, i2, g, g), reps=3), nbytes=2.0 * 256 * 8192 * 56),
    }
    del c, cen, p, d1, d2, i1, i2, g
    # ---- C5: scene scale, one cloud per GPU, unsharded form
    c = cloud(1, 100000, 6)
    cen = ops.fps_gather(c, 2048)[1]
    p = c + 0.01 * torch.randn_like(c)
    out["C5 N=100000 G=2048 M=64 (one GPU, unsharded)"] = {
        "fps 100k->2048": entry(_median_ms(lambda: ops.fps_gather(c, 2048), reps=3)),
        "group k=64": entry(_median_ms(lambda: ops.group_points_knn(c, cen, 64, want_idx=False), reps=3), pairs=2048.0 * 100000),
        "chamfer fwd 100k^2": entry(_median_ms(lambda: ops.chamfer_forward(p, c), reps=3), pairs=2.0 * 100000 * 100000),
    }
    return out


def sharded_c5_block(dev, world, rank, max_over_ranks):
    """BASELINE config 5 with the Chamfer / kNN reference set sharded over the ranks (SURVEY.md 8e): Chamfer forward +
    backward and kNN at N = 100 000 over NCCL, bit-exactness against the unsharded kernels on the same GPU, and the
    share of the sharded time spent outside the local kernels (the collective + its launch)."""
    import torch
    import torch.distributed as dist
    from pointdae_b200 import ops, sharded, synth

    n, q, k = 100000, 2048, 64
    xyz2 = torch.from_numpy(synth.adversarial(synth.clouds(1, n, seed=5), seed=5, n_small=0, n_dup=200)).to(dev)
    xyz1 = torch.from_numpy(synth.prediction(synth.clouds(1, n, seed=5), seed=5)).to(dev)
    lo, hi = sharded.shard_bounds(n, world, rank)
    local_refs = xyz2[:, lo:hi].contiguous()

    def synced_ms(fn, reps=10):
        for _ in range(3):
            fn()
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return max_over_ranks(a.elapsed_time(b) / reps)

    def all_ok(flag):
        t = torch.tensor([1 if flag else 0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    # exchange forms: the fused peer-memory kernel (default when symmetric memory is available), its in-switch (NVLS)
    # variant, and the NCCL all-reduce it replaces
    forms = {"nccl_all_reduce": None}
    for nm, mm in (("peer_kernel", False), ("multimem_kernel", True)):
        ex = sharded.make_exchange(n, dev, use_multimem=mm)
        if ex is not None and (ex.use_multimem == mm):
            forms[nm] = ex
    best = "multimem_kernel" if "multimem_kernel" in forms else ("peer_kernel" if "peer_kernel" in forms else "nccl_all_reduce")
    exchange = forms[best]
    out = {"n_points": n, "world": world, "impl": sharded.exchange_name(exchange), "exchange_forms_ms": {}}
    for nm, ex in forms.items():
        t = synced_ms(lambda: sharded.chamfer_forward_sharded(xyz1, local_refs, lo, exchange=ex))
        r = sharded.chamfer_forward_sharded(xyz1, local_refs, lo, exchange=ex)
        out["exchange_forms_ms"][nm] = {"forward_ms": t, "name": sharded.exchange_name(ex)}
        out["exchange_forms_ms"][nm]["_res"] = [x.clone() for x in r]
    ref_res = out["exchange_forms_ms"]["nccl_all_reduce"]["_res"]
    for nm in list(out["exchange_forms_ms"]):
        res = out["exchange_forms_ms"][nm].pop("_res")
        out["exchange_forms_ms"][nm]["same_bits_as_nccl_form"] = all_ok(all(torch.equal(a, bb) for a, bb in zip(res, ref_res)))
    fwd_ms = out["exchange_forms_ms"][best]["forward_ms"]
    local_ms = synced_ms(lambda: ops.chamfer_unpack_keys(ops.chamfer_sharded_local(xyz1, local_refs, lo)[0]))
    unsharded_ms = _median_ms(lambda: ops.chamfer_forward(xyz1, xyz2), reps=5)
    d1, d2l, i1, i2l = [x.clone() for x in sharded.chamfer_forward_sharded(xyz1, local_refs, lo, exchange=exchange)]
    fd1, fd2, fi1, fi2 = ops.chamfer_forward(xyz1, xyz2)
    ok = torch.equal(d1, fd1) and torch.equal(i1, fi1) and torch.equal(d2l, fd2[:, lo:hi]) and torch.equal(i2l, fi2[:, lo:hi])
    out["chamfer_forward"] = {"sharded_ms": fwd_ms, "local_kernels_only_ms": local_ms,
                              "exchange_share": max(0.0, 1.0 - local_ms / fwd_ms), "unsharded_1gpu_ms": max_over_ranks(unsharded_ms),
                              "speedup_vs_1gpu": max_over_ranks(unsharded_ms) / fwd_ms,
                              "efficiency_vs_1gpu": max_over_ranks(unsharded_ms) / fwd_ms / world,
                              "bit_exact_vs_unsharded": all_ok(ok),
                              "fma_pipe_frac_algorithmic_all_gpus": 2.0 * n * n * 6 / (fwd_ms * 1e-3) / (world * 148 * 128 * 1.965e9)}
    g1 = torch.full_like(fd1, 1.0 / fd1.numel())
    g2 = torch.full_like(fd2, 1.0 / fd2.numel())
    g2l = g2[:, lo:hi].contiguous()
    bwd_ms = synced_ms(lambda: sharded.chamfer_backward_sharded(xyz1, local_refs, lo, i1, i2l, g1, g2l))
    gx1, gx2l = sharded.chamfer_backward_sharded(xyz1, local_refs, lo, i1, i2l, g1, g2l)
    w1, w2 = ops.chamfer_backward(xyz1, xyz2, fi1, fi2, g1, g2)
    ok_b = (torch.allclose(gx1, w1, rtol=1e-5, atol=1e-6 * float(w1.abs().max()))
            and torch.allclose(gx2l, w2[:, lo:hi], rtol=1e-5, atol=1e-6 * float(w2.abs().max())))
    bwd2_ms = synced_ms(lambda: sharded.chamfer_backward_gathered(xyz1, local_refs, lo, n, i1, i2l, g1, g2l))
    hx1, hx2l = sharded.chamfer_backward_gathered(xyz1, local_refs, lo, n, i1, i2l, g1, g2l)
    ok_b2 = (torch.allclose(hx1, w1, rtol=1e-5, atol=1e-6 * float(w1.abs().max()))
             and torch.allclose(hx2l, w2[:, lo:hi], rtol=1e-5, atol=1e-6 * float(w2.abs().max())))
    out["chamfer_backward"] = {"masked_all_reduce_ms": bwd_ms, "matches_unsharded_1e-5": all_ok(ok_b),
                               "gathered_ms": bwd2_ms, "gathered_matches_unsharded_1e-5": all_ok(ok_b2),
                               "unsharded_1gpu_ms": max_over_ranks(_median_ms(lambda: ops.chamfer_backward(xyz1, xyz2, fi1, fi2, g1, g2)))}
    centers = ops.fps_gather(xyz2, q)[1]
    knn_ms = synced_ms(lambda: sharded.knn_sharded(local_refs, centers, k, lo))
    knn_local_ms = synced_ms(lambda: ops.knn_keys(local_refs, centers, k, lo))
    knn_1gpu = _median_ms(lambda: ops.knn_points(xyz2, centers, k), reps=5)
    kd, ki = sharded.knn_sharded(local_refs, centers, k, lo)
    wd, wi = ops.knn_points(xyz2, centers, k)
    out["knn"] = {"queries": q, "k": k, "sharded_ms": knn_ms, "local_kernel_only_ms": knn_local_ms,
                  "exchange_share": max(0.0, 1.0 - knn_local_ms / knn_ms), "unsharded_1gpu_ms": max_over_ranks(knn_1gpu),
                  "speedup_vs_1gpu": max_over_ranks(knn_1gpu) / knn_ms,
                  "bit_exact_vs_unsharded": all_ok(torch.equal(kd, wd) and torch.equal(ki, wi))}
    return out


def other_kernels(dev, clouds_d, preds_d, peaks, props):
    """SURVEY.md 8(d): the path's other kernels, each timed alone with CUDA events over replayed graphs (outside the
    timed region): FPS as us per sequential iteration, the 3-D kNN against the FP32 FMA pipe, graph feature and the
    Chamfer backward against the measured HBM copy peak.  Evidence only; a failure here never breaks the bench line."""
    import torch
    from pointdae_b200 import dgcnn_util, ops, synth

    def eager_us(fn, reps=10):  # long kernels: launch overhead is noise, no capture needed
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e3 / reps

    def timed_us(fn, reps=40):
        fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            keep = [fn() for _ in range(4)]
        g.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            g.replay()
        b.record()
        torch.cuda.synchronize()
        del keep
        return a.elapsed_time(b) * 1e3 / (4 * reps)

    out = {}
    hbm = float(peaks.get("hbm_gbs", 6556.5))
    fma = props.multi_processor_count * 128 * float(peaks.get("sm_max_mhz", 1965.0)) * 1e6  # lane-ops / s
    c, p = clouds_d[0], preds_d[0]
    t = timed_us(lambda: ops.fps_gather(c, G))
    out["fps+centre gather %dx%d->%d" % (B, N, G)] = {"us": t, "us_per_iteration": t / (G - 1), "bound": "latency (one CTA per cloud, %d of %d SMs)" % (min(B, props.multi_processor_count), props.multi_processor_count)}
    center = ops.fps_gather(c, G)[1]
    t = timed_us(lambda: ops.group_points_knn(c, center, M, want_idx=False))
    out["group kNN %d + gather" % M] = {"us": t, "fma_pipe_frac_algorithmic": B * G * N * 6.0 / (t * 1e-6) / fma,
                                    "bound": "per-warp latency + instruction issue of the selection at this size (16.8 M pairs = "
                                             "2.7 us of FMA work); see `configs` for the shapes where the FMA pipe binds"}
    t = timed_us(lambda: ops.fps_group(c, G, M, want_idx=False))
    t_fps = out["fps+centre gather %dx%d->%d" % (B, N, G)]["us"]
    out["patchifier, one launch (fps + group kNN %d)" % M] = {
        "us": t, "us_after_the_last_fps_iteration": t - t_fps,
        "bound": "FPS latency: the search of centre j runs on consumer warps of the same CTA beside FPS iterations j+1.. "
                 "(csrc/patchify.cu); the two-launch form costs the sum of the two entries above"}
    d1, d2, i1, i2 = ops.chamfer_forward(p, c)
    gone = torch.ones(1, device=dev)
    t = timed_us(lambda: ops.chamfer_loss_backward(p, c, i1, i2, d1, d2, gone, 1.0, 1.0))
    tl = timed_us(lambda: ops.chamfer_mean_loss(d1, d2))
    out["chamfer mean loss (2 launches)"] = {"us": tl, "bound": "launch latency (128 partial sums + ordered fp64 final sum)"}
    out["chamfer backward (2 launches)"] = {"us": t, "GBps": 2 * B * N * 56 / (t * 1e-6) / 1e9, "hbm_frac": 2 * B * N * 56 / (t * 1e-6) / 1e9 / hbm,
                                           "bound": "L2 atomics / launch latency (56 B per point, L2 resident)"}
    Cf, Bf, kf = 128, 16, 20
    x = torch.from_numpy(synth.features(Bf, Cf, N, seed=Cf)).to(dev)
    t = eager_us(lambda: dgcnn_util.knn(x, kf))
    out["dgcnn knn C=%d k=%d %dx%d" % (Cf, kf, Bf, N)] = {"us": t, "fma_pipe_frac": Bf * N * N * Cf * 1.0 / (t * 1e-6) / fma,
                                                       "bound": "FP32 FMA pipe (direct form, 2C flop per pair)"}
    idx = dgcnn_util.knn(x, kf)
    t = eager_us(lambda: ops._graph_feature_fwd(x, idx))
    nbytes = Bf * N * kf * 2 * Cf * 4 + Bf * Cf * N * 4 + Bf * N * kf * 8
    out["graph feature C=%d" % Cf] = {"us": t, "GBps": nbytes / (t * 1e-6) / 1e9, "hbm_frac": nbytes / (t * 1e-6) / 1e9 / hbm,
                                      "bound": "HBM write stream", "peak_GBps": hbm}
    return out


STEP_OUTPUTS = ("neighborhood", "center", "fps_idx", "dist1", "dist2", "idx1", "idx2", "loss3", "gpred", "gcloud")


def dump_outputs(out_dir, out):
    """Writes the outputs of one timed step as out_dir/<name>.npy so that two builds can be compared array for array:
    the StepBuffers of the native step call, or (loss, neighborhood, gpred) of the graph / eager arms.  Floating
    arrays are stored as float32, index arrays as float64 (exact).  At the headline shape this is about 16 MB."""
    import numpy as np
    if isinstance(out, tuple):
        arrays = dict(zip(("loss", "neighborhood", "gpred"), out))
    else:
        arrays = {name: getattr(out, name) for name in STEP_OUTPUTS}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


_REAL_STDOUT = None


def emit(line):
    """the one JSON line, written to the process's original stdout"""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries (NCCL's version banner, torch warnings) may print to stdout; the contract is ONE JSON line there.
    # Keep a private handle on the real stdout and point fd 1 at stderr for everything else.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-gpu", action="store_true", help="skip timing the reference's own CUDA ops (oracle/_ref)")
    ap.add_argument("--sched", default="torch", choices=["torch", "priority"],
                    help="priority: graphs instantiated with per-node launch priorities (Chamfer branch first)")
    ap.add_argument("--launch", default="native", choices=["graph", "native"],
                    help="resident arm: graph = the step captured from the Python op layer and replayed as a CUDA graph; "
                         "native = one pdae_step_f32 call per step (the same six launches issued from C++, no graph)")
    ap.add_argument("--patchify", default="fused", choices=["fused", "two"],
                    help="fused: FPS + Group as one launch (pdae_fps_group_f32); two: pdae_fps_gather_f32 + pdae_group_ws_f32")
    ap.add_argument("--patchifier", default="tail", choices=["tail", "pdl", "tail2", "split", "first", "overlap"],
                    help="where FPS + Group run relative to the Chamfer forward: beside the loss / backward kernels after it "
                         "(default), before it (the model's order), or from the start on a second stream (round 1)")
    ap.add_argument("--knn-gate", default="none", choices=["scan", "none"],
                    help="none: both branches start together (default, fastest); scan: the patchifier's kNN waits for "
                         "the Chamfer scan kernel and overlaps the step's tail instead (measured 6 %% slower: the tail "
                         "kernels are issue-bound like the kNN, the FMA-bound scan is the better partner)")
    ap.add_argument("--no-graphs", action="store_true", help="issue the resident chain eagerly instead of replaying CUDA graphs")
    ap.add_argument("--e2e-upload", default="cloud", choices=["cloud", "both"],
                    help="what the end-to-end arm copies from pinned host memory every step: the cloud (default; the "
                         "prediction is produced on the device by the model) or cloud + prediction")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config (C2..C5) and sharded-C5 evidence blocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (rank 0; the inputs "
                         "depend only on the arguments, so two builds run with the same arguments can be compared)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm (the CPU reference arm sizes its batch by wall-clock time)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
