"""ctypes front ends of oracle/pdae_oracle_det.c: the deterministic gradients in their defined summation order, fp32,
bit for bit what the *_det entry points of the library compute.  Same build flags as oracle/cpu.py."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pdae_oracle_det.c")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libpdae_oracle_det.so")
_lib = None


def build(force=False):
    """gcc -O2 -ffp-contract=off (no implicit fusion) -> oracle/_build/libpdae_oracle_det.so"""
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


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def chamfer_bwd(xyz1, xyz2, idx1, idx2, gd1, gd2):
    """xyz read as (B, N, 3) rows like the kernels; -> grad_xyz1 (B,N,3), grad_xyz2 (B,M,3)."""
    xyz1, xyz2 = _f32(xyz1), _f32(xyz2)
    idx1, idx2, gd1, gd2 = _i32(idx1), _i32(idx2), _f32(gd1), _f32(gd2)
    b, n = idx1.shape
    m = idx2.shape[1]
    g1 = np.empty((b, n, 3), dtype=np.float32)
    g2 = np.empty((b, m, 3), dtype=np.float32)
    lib().pdae_oracle_chamfer_bwd_ordered(_p(xyz1), _p(xyz2), _p(idx1), _p(idx2), _p(gd1), _p(gd2), b, n, m, _p(g1), _p(g2))
    return g1, g2


def chamfer_loss_grad_arrays(gloss, w1, w2, b, n, m, dist1=None, dist2=None):
    """The per-point d(loss)/d(dist) that the fused mean-loss backward forms (chamfer.cu GradMean), in the same fp32
    operations: gloss * rn(w / count), and for L1 (dists given) divided by 2 sqrt(dist)."""
    g = np.float32(gloss)
    out = []
    for w, cnt, d in ((w1, b * n, dist1), (w2, b * m, dist2)):
        s = np.float32(np.float32(w) / np.float32(cnt)) * g
        if d is None:
            out.append(np.full((b, cnt // b), s, dtype=np.float32))
        else:
            with np.errstate(divide="ignore", invalid="ignore"):
                out.append((s / (np.float32(2.0) * np.sqrt(_f32(d)))).astype(np.float32))
    return out


def gather_grad(gout, idx, n):
    gout, idx = _f32(gout), _i32(idx)
    b, c, m = gout.shape
    g = np.empty((b, c, int(n)), dtype=np.float32)
    lib().pdae_oracle_gather_grad_ordered(_p(gout), _p(idx), b, c, int(n), m, _p(g))
    return g


def group_points_grad(gout, idx, n):
    gout, idx = _f32(gout), _i32(idx)
    b, c, p, s = gout.shape
    g = np.empty((b, c, int(n)), dtype=np.float32)
    lib().pdae_oracle_group_points_grad_ordered(_p(gout), _p(idx), b, c, int(n), p, s, _p(g))
    return g


def three_interpolate_grad(gout, idx, weight, m):
    gout, idx, weight = _f32(gout), _i32(idx), _f32(weight)
    b, c, n = gout.shape
    g = np.empty((b, c, int(m)), dtype=np.float32)
    lib().pdae_oracle_three_interpolate_grad_ordered(_p(gout), _p(idx), _p(weight), b, c, n, int(m), _p(g))
    return g


def graph_feature_grad(gout_phys, idx):
    """gout physical (B,N,k,2C) -> gx (B,C,N)."""
    g = _f32(gout_phys)
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    b, n, k, c2 = g.shape
    c = c2 // 2
    gx = np.empty((b, c, n), dtype=np.float32)
    lib().pdae_oracle_graph_feature_grad_ordered(_p(g), _p(idx), b, c, n, k, _p(gx))
    return gx


def reverse_index(idx, t):
    """numpy reference of pdae_reverse_index_*: per cloud, ptr (t+1) and the stable argsort of the in-range targets."""
    idx = np.asarray(idx)
    b, s = idx.shape
    ptr = np.zeros((b, t + 1), dtype=np.int32)
    slots = []
    for i in range(b):
        row = idx[i].astype(np.int64)
        ok = (row >= 0) & (row < t)
        ptr[i, 1:] = np.cumsum(np.bincount(row[ok], minlength=t))
        j = np.nonzero(ok)[0]
        slots.append(j[np.argsort(row[ok], kind="stable")].astype(np.int32))
    return ptr, slots
