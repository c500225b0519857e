"""ctypes front ends of oracle/pdae_oracle_pointops.c: segment FPS and segment kNN of packed variable-size clouds in
the kernels' fp32 operations and tie rules, plus float64 transcriptions of the published pointops loops (the literal
block tree and the literal per-thread heap) that check the oracle.  Same build flags as oracle/cpu.py."""
import ctypes
import math
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pdae_oracle_pointops.c")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libpdae_oracle_pointops.so")
_lib = None


def build(force=False):
    """gcc -O2 -ffp-contract=off (no implicit fusion) -> oracle/_build/libpdae_oracle_pointops.so"""
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= os.path.getmtime(SRC):
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-std=gnu11", "-o", LIB,
                           SRC, "-lm"])
    return LIB


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(SRC):
            build()
        _lib = ctypes.CDLL(LIB)
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def block_size(n):
    return int(lib().pdae_oracle_seg_fps_block_size(int(n)))


def largest(offset):
    off = np.asarray(offset, np.int64)
    return int(np.diff(off, prepend=0).max()) if off.size else 0


def seg_fps(xyz, offset, new_offset, n=None, m=None, tmp=None):
    """-> (idx (m,) int32, tmp after the call (N,) fp32, or None when tmp was None).  n defaults to the largest
    segment and m to new_offset[-1], as ops.segment_fps does."""
    xyz, offset, new_offset = _f32(xyz).reshape(-1, 3), _i32(offset), _i32(new_offset)
    n = largest(offset) if n is None else int(n)
    m = (int(new_offset[-1]) if new_offset.size else 0) if m is None else int(m)
    idx = np.full(max(m, 0), -7, dtype=np.int32)  # -7: a slot no sample writes stays visible
    t = _f32(tmp).copy() if tmp is not None else None
    scratch = np.empty(max(xyz.shape[0], 1), dtype=np.float32)
    lib().pdae_oracle_seg_fps(_p(xyz), xyz.shape[0], _p(offset), _p(new_offset), offset.size, n, idx.size, _p(t), _p(idx),
                              _p(scratch))
    return idx, t


def seg_knn(nsample, xyz, new_xyz, offset, new_offset):
    """-> (idx (M,nsample) int32, dist2 (M,nsample) fp32)"""
    xyz, new_xyz = _f32(xyz).reshape(-1, 3), _f32(new_xyz).reshape(-1, 3)
    offset, new_offset = _i32(offset), _i32(new_offset)
    m = new_xyz.shape[0]
    idx = np.empty((m, nsample), dtype=np.int32)
    d2 = np.empty((m, nsample), dtype=np.float32)
    lib().pdae_oracle_seg_knn(_p(xyz), xyz.shape[0], _p(new_xyz), m, _p(offset), _p(new_offset), offset.size, int(nsample),
                              _p(idx), _p(d2))
    return idx, d2


# ------------------------------------------------------------------ float64 transcriptions of the published loops
def fps_published_f64(xyz, offset, new_offset, n, tmp=None):
    """furthestsampling_cuda_kernel, one block per segment, in float64: every thread's strided loop with its strict
    `>` from best = -1, then the shared-memory tree whose __update keeps the lower slot on ties.
    -> (idx (m,) int64, tmp (N,) float64)"""
    xyz = np.asarray(xyz, np.float64).reshape(-1, 3)
    pow_2 = int(math.log(float(n)) / math.log(2.0)) if n > 0 else 0
    bs = max(min(1 << pow_2, 1024), 1)
    t = np.full(xyz.shape[0], 1e10) if tmp is None else np.asarray(tmp, np.float64).copy()
    m = int(new_offset[-1])
    idx = np.full(m, -7, dtype=np.int64)
    for s in range(len(offset)):
        sn, en = (int(offset[s - 1]) if s else 0), int(offset[s])
        sm, em = (int(new_offset[s - 1]) if s else 0), int(new_offset[s])
        if em <= sm:
            continue
        idx[sm] = sn
        old = sn
        for j in range(sm + 1, em):
            d = ((xyz[sn:en] - xyz[old]) ** 2).sum(-1)
            t[sn:en] = np.minimum(d, t[sn:en])
            # thread tid: for (k = start_n + tid; k < end_n; k += stride) with a strict `>` from best = -1, i.e. the
            # first maximum of its column when that exceeds -1, else (-1, start_n)
            rows = max(-(-(en - sn) // bs), 1)
            cols = np.full(rows * bs, -np.inf)
            cols[:en - sn] = t[sn:en]
            cols = cols.reshape(rows, bs)
            top, first = cols.max(0), cols.argmax(0)
            taken = top > -1.0
            dists = np.where(taken, top, -1.0)
            dists_i = np.where(taken, sn + np.arange(bs) + first * bs, sn).astype(np.int64)
            stride = bs // 2
            while stride >= 1:  # __update(dists, dists_i, tid, tid + stride) for tid < stride
                v1, v2 = dists[:stride].copy(), dists[stride:2 * stride]
                i1, i2 = dists_i[:stride].copy(), dists_i[stride:2 * stride]
                dists[:stride] = np.maximum(v1, v2)
                dists_i[:stride] = np.where(v2 > v1, i2, i1)
                stride //= 2
            old = int(dists_i[0])
            idx[j] = old
    return idx, t


def _reheap(dist, idx, k):
    root, child = 0, 1
    while child < k:
        if child + 1 < k and dist[child + 1] > dist[child]:
            child += 1
        if dist[root] > dist[child]:
            return
        dist[root], dist[child] = dist[child], dist[root]
        idx[root], idx[child] = idx[child], idx[root]
        root = child
        child = root * 2 + 1


def _heap_sort(dist, idx, k):
    for i in range(k - 1, 0, -1):
        dist[0], dist[i] = dist[i], dist[0]
        idx[0], idx[i] = idx[i], idx[0]
        _reheap(dist, idx, i)


def knn_published_f64(nsample, xyz, new_xyz, offset, new_offset):
    """knnquery_cuda_kernel in float64 with its literal max-heap (reheap / heap_sort), rows the offsets cover.
    -> (idx (M,nsample) int64, dist2 (M,nsample) float64); rows past new_offset[-1] are left at (-7, nan)."""
    xyz = np.asarray(xyz, np.float64).reshape(-1, 3)
    new_xyz = np.asarray(new_xyz, np.float64).reshape(-1, 3)
    m = new_xyz.shape[0]
    out_i = np.full((m, nsample), -7, dtype=np.int64)
    out_d = np.full((m, nsample), np.nan)
    for pt in range(min(m, int(new_offset[-1]))):
        bt = 0
        while not pt < int(new_offset[bt]):  # get_bt_idx
            bt += 1
        start = int(offset[bt - 1]) if bt else 0
        end = int(offset[bt])
        best_dist = [1e10] * nsample
        best_idx = [start] * nsample
        q = new_xyz[pt]
        d2s = ((xyz[start:end] - q) ** 2).sum(-1)
        for i in range(start, end):
            d2 = float(d2s[i - start])
            if d2 < best_dist[0]:
                best_dist[0] = d2
                best_idx[0] = i
                _reheap(best_dist, best_idx, nsample)
        _heap_sort(best_dist, best_idx, nsample)
        out_i[pt], out_d[pt] = best_idx, best_dist
    return out_i, out_d
