"""ctypes front ends of oracle/pdae_oracle_emd.c: the approximate Earth Mover's Distance in the kernels' fp32 operations
and orders (libm exp2f / 1 / sqrtf in place of ex2.approx / rsqrtf).  Same build flags as oracle/cpu.py."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "pdae_oracle_emd.c")
OUT_DIR = os.path.join(HERE, "_build")
LIB = os.path.join(OUT_DIR, "libpdae_oracle_emd.so")
LEVELS = 10
_lib = None


def build(force=False):
    """gcc -O2 -ffp-contract=off (no implicit fusion) -> oracle/_build/libpdae_oracle_emd.so"""
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


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def match(xyz1, xyz2, accumulate=True):
    """xyz1 (B,n,3), xyz2 (B,m,3) -> ratio_l (B,10,n), ratio_r (B,10,m) and, with accumulate, the match (B,m,n)
    accumulated level by level like the published kernel (else None)."""
    xyz1, xyz2 = _f32(xyz1), _f32(xyz2)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    rl = np.empty((b, LEVELS, n), dtype=np.float32)
    rr = np.empty((b, LEVELS, m), dtype=np.float32)
    mt = np.empty((b, m, n), dtype=np.float32) if accumulate else None
    scratch = np.empty(n + m, dtype=np.float32)
    lib().pdae_oracle_emd_match(_p(xyz1), _p(xyz2), b, n, m, _p(rl), _p(rr), _p(mt) if accumulate else None, _p(scratch))
    return rl, rr, mt


def rebuild(xyz1, xyz2, ratio_l, ratio_r):
    """the match (B,m,n) from the per-level ratios, in the kernels' expression and level order"""
    xyz1, xyz2, ratio_l, ratio_r = _f32(xyz1), _f32(xyz2), _f32(ratio_l), _f32(ratio_r)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    mt = np.empty((b, m, n), dtype=np.float32)
    lib().pdae_oracle_emd_rebuild(_p(xyz1), _p(xyz2), b, n, m, _p(ratio_l), _p(ratio_r), _p(mt))
    return mt


def cost(xyz1, xyz2, match_):
    xyz1, xyz2, match_ = _f32(xyz1), _f32(xyz2), _f32(match_)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    out = np.empty(b, dtype=np.float32)
    lib().pdae_oracle_emd_cost(_p(xyz1), _p(xyz2), b, n, m, _p(match_), _p(out))
    return out


def grad(grad_cost, xyz1, xyz2, match_):
    grad_cost, xyz1, xyz2, match_ = _f32(grad_cost), _f32(xyz1), _f32(xyz2), _f32(match_)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    g1 = np.empty((b, n, 3), dtype=np.float32)
    g2 = np.empty((b, m, 3), dtype=np.float32)
    lib().pdae_oracle_emd_grad(_p(grad_cost), _p(xyz1), _p(xyz2), b, n, m, _p(match_), _p(g1), _p(g2))
    return g1, g2


def match_f64(xyz1, xyz2):
    """Plain float64 numpy transcription of the published loop (exp, no ordering): the oracle's own check.
    -> match (B,m,n) float64"""
    xyz1, xyz2 = np.asarray(xyz1, np.float64), np.asarray(xyz2, np.float64)
    b, n, _ = xyz1.shape
    m = xyz2.shape[1]
    out = np.zeros((b, m, n))
    for bi in range(b):
        d = ((xyz2[bi][:, None, :] - xyz1[bi][None, :, :]) ** 2).sum(-1)  # (m, n): [l][k]
        reml = np.full(n, 1.0 if n >= m else float(m // n))
        remr = np.full(m, float(n // m) if n >= m else 1.0)
        for j in range(7, -3, -1):
            e = np.exp((-(4.0 ** j) if j > -2 else 0.0) * d)
            ratio_l = reml / (1e-9 + (e * remr[:, None]).sum(0))
            sumr = (e * ratio_l[None, :]).sum(1) * remr
            ratio_r = np.minimum(remr / (sumr + 1e-9), 1.0) * remr
            remr = np.maximum(0.0, remr - sumr)
            w = e * ratio_l[None, :] * ratio_r[:, None]
            out[bi] += w
            reml = np.maximum(0.0, reml - w.sum(0))
    return out


def cost_f64(xyz1, xyz2, match_):
    xyz1, xyz2 = np.asarray(xyz1, np.float64), np.asarray(xyz2, np.float64)
    d = np.sqrt(((xyz2[:, :, None, :] - xyz1[:, None, :, :]) ** 2).sum(-1))
    return (d * match_).sum((1, 2))
