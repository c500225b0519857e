"""CPU oracle of the segment EMD (csrc/segemd.cu): a loop over segments of the equal-size EMD oracle at b = 1
(cpu_emd.match / rebuild / cost / grad), the packed level-major ratio layout, and the rules for segments with an empty
side and points past the last segment (ratios, cost and gradients 0).  numpy only; no build step of its own (the
oracle it calls is built by cpu_emd.build())."""
import numpy as np

from . import cpu_emd
from .cpu_segchamfer import segments

LEVELS = cpu_emd.LEVELS


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _pairs(xyz1, xyz2, offset1, offset2):
    """(s, lo1, hi1, lo2, hi2) of the segments whose two sides both hold points"""
    for s, (lo1, hi1, lo2, hi2) in enumerate(segments(offset1, offset2, len(xyz1), len(xyz2))):
        if hi1 > lo1 and hi2 > lo2:
            yield s, lo1, hi1, lo2, hi2


def match(xyz1, xyz2, offset1, offset2):
    """-> ratio_l (10,N), ratio_r (10,M) f32, level-major, and {s: match (m_s, n_s)} of the segments with both sides"""
    xyz1, xyz2 = _f32(xyz1), _f32(xyz2)
    rl = np.zeros((LEVELS, len(xyz1)), np.float32)
    rr = np.zeros((LEVELS, len(xyz2)), np.float32)
    mats = {}
    for s, lo1, hi1, lo2, hi2 in _pairs(xyz1, xyz2, offset1, offset2):
        a, b, mt = cpu_emd.match(xyz1[None, lo1:hi1], xyz2[None, lo2:hi2])
        rl[:, lo1:hi1], rr[:, lo2:hi2], mats[s] = a[0], b[0], mt[0]
    return rl, rr, mats


def _rebuild(xyz1, xyz2, ratio_l, ratio_r, lo1, hi1, lo2, hi2):
    return cpu_emd.rebuild(xyz1[None, lo1:hi1], xyz2[None, lo2:hi2], _f32(ratio_l)[None, :, lo1:hi1],
                           _f32(ratio_r)[None, :, lo2:hi2])


def cost(xyz1, xyz2, offset1, offset2, ratio_l, ratio_r):
    """-> (b,) f32 from the match rebuilt from the given ratios; 0 for a segment with an empty side"""
    xyz1, xyz2 = _f32(xyz1), _f32(xyz2)
    out = np.zeros(len(np.asarray(offset1)), np.float32)
    for s, lo1, hi1, lo2, hi2 in _pairs(xyz1, xyz2, offset1, offset2):
        mt = _rebuild(xyz1, xyz2, ratio_l, ratio_r, lo1, hi1, lo2, hi2)
        out[s] = cpu_emd.cost(xyz1[None, lo1:hi1], xyz2[None, lo2:hi2], mt)[0]
    return out


def grad(grad_cost, xyz1, xyz2, offset1, offset2, ratio_l, ratio_r):
    """-> grad1 (N,3), grad2 (M,3) f32 with the match rebuilt from the given ratios held constant; 0 for points of a
    segment with an empty side and past the last segment"""
    xyz1, xyz2 = _f32(xyz1), _f32(xyz2)
    gc = _f32(grad_cost)
    g1, g2 = np.zeros((len(xyz1), 3), np.float32), np.zeros((len(xyz2), 3), np.float32)
    for s, lo1, hi1, lo2, hi2 in _pairs(xyz1, xyz2, offset1, offset2):
        mt = _rebuild(xyz1, xyz2, ratio_l, ratio_r, lo1, hi1, lo2, hi2)
        a, b = cpu_emd.grad(gc[s:s + 1], xyz1[None, lo1:hi1], xyz2[None, lo2:hi2], mt)
        g1[lo1:hi1], g2[lo2:hi2] = a[0], b[0]
    return g1, g2
