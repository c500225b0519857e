"""CPU oracle of the segment Chamfer distance (csrc/segchamfer.cu): a loop over segments of the equal-size oracles at
b = 1 (cpu.chamfer_fwd, and cpu_det.chamfer_bwd for the ordered gradient), the global-index shift, the rules for
points without an opposite segment, and the cloud-weighted mean losses in float64.  numpy only; no build step of its
own (the two oracles it calls are built by cpu.build() / cpu_det.build())."""
import numpy as np

from . import cpu, cpu_det


def ends(offset, total):
    """end[s] = max(clamp(offset[0..s], 0, total)): row p belongs to the first segment s with p < offset[s]."""
    o = np.clip(np.asarray(offset, dtype=np.int64), 0, total)
    return np.maximum.accumulate(o) if o.size else o


def segments(offset1, offset2, n, m):
    """[(lo1, hi1, lo2, hi2)] per segment"""
    e1, e2 = ends(offset1, n), ends(offset2, m)
    s1, s2 = np.concatenate(([0], e1[:-1])), np.concatenate(([0], e2[:-1]))
    return [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(s1, e1, s2, e2)]


def fwd(xyz1, xyz2, offset1, offset2):
    """-> dist1 (N,), dist2 (M,) f32, idx1, idx2 int32 global; (0, -1) where a point has no opposite segment."""
    xyz1 = np.ascontiguousarray(xyz1, dtype=np.float32)
    xyz2 = np.ascontiguousarray(xyz2, dtype=np.float32)
    n, m = len(xyz1), len(xyz2)
    d1, d2 = np.zeros(n, np.float32), np.zeros(m, np.float32)
    i1, i2 = np.full(n, -1, np.int32), np.full(m, -1, np.int32)
    for lo1, hi1, lo2, hi2 in segments(offset1, offset2, n, m):
        if hi1 > lo1 and hi2 > lo2:
            a, b, c, d = cpu.chamfer_fwd(xyz1[None, lo1:hi1], xyz2[None, lo2:hi2])
            d1[lo1:hi1], d2[lo2:hi2] = a[0], b[0]
            i1[lo1:hi1], i2[lo2:hi2] = c[0] + lo2, d[0] + lo1
    return d1, d2, i1, i2


def bwd(xyz1, xyz2, idx1, idx2, gd1, gd2, offset1, offset2):
    """Ordered gradient (own term, then the points that chose this one, ascending): -> gx1 (N,3), gx2 (M,3)."""
    xyz1 = np.ascontiguousarray(xyz1, dtype=np.float32)
    xyz2 = np.ascontiguousarray(xyz2, dtype=np.float32)
    n, m = len(xyz1), len(xyz2)
    g1, g2 = np.zeros((n, 3), np.float32), np.zeros((m, 3), np.float32)
    gd1, gd2 = np.asarray(gd1, np.float32), np.asarray(gd2, np.float32)
    for lo1, hi1, lo2, hi2 in segments(offset1, offset2, n, m):
        if hi1 > lo1 and hi2 > lo2:
            a, b = cpu_det.chamfer_bwd(xyz1[None, lo1:hi1], xyz2[None, lo2:hi2], (idx1[lo1:hi1] - lo2)[None],
                                       (idx2[lo2:hi2] - lo1)[None], gd1[None, lo1:hi1], gd2[None, lo2:hi2])
            g1[lo1:hi1], g2[lo2:hi2] = a[0], b[0]
    return g1, g2


def loss_f64(dist1, dist2, offset1, offset2, l1=False):
    """-> (loss, term1, term2, |S|) in float64 from the fp32 distances."""
    d1, d2 = np.asarray(dist1, np.float64), np.asarray(dist2, np.float64)
    t1 = t2 = 0.0
    ns = 0
    for lo1, hi1, lo2, hi2 in segments(offset1, offset2, len(d1), len(d2)):
        if hi1 > lo1 and hi2 > lo2:
            a, b = d1[lo1:hi1], d2[lo2:hi2]
            if l1:
                a, b = np.sqrt(a), np.sqrt(b)
            t1, t2, ns = t1 + a.mean(), t2 + b.mean(), ns + 1
    if ns == 0:
        return 0.0, 0.0, 0.0, 0
    t1, t2 = t1 / ns, t2 / ns
    return ((t1 + t2) / 2 if l1 else t1 + t2), t1, t2, ns


def loss_grad_arrays(gloss, dist1, dist2, offset1, offset2, l1=False):
    """The per-point d(loss)/d(dist) of the fused loss backward in its fp32 operations: gloss * rn(w / (|S| * size_s)),
    divided by 2 sqrt(dist) for L1; 0 for points outside S."""
    d1, d2 = np.asarray(dist1, np.float32), np.asarray(dist2, np.float32)
    segs = [s for s in segments(offset1, offset2, len(d1), len(d2)) if s[1] > s[0] and s[3] > s[2]]
    w = np.float32(0.5 if l1 else 1.0)
    g = np.float32(gloss)
    out = []
    for side, d in ((0, d1), (1, d2)):
        a = np.zeros(len(d), np.float32)
        for s in segs:
            lo, hi = s[2 * side], s[2 * side + 1]
            wt = np.float32(w / np.float32(len(segs) * (hi - lo)))
            v = np.full(hi - lo, g * wt, np.float32)
            if l1:
                with np.errstate(divide="ignore", invalid="ignore"):
                    v = (v / (np.float32(2.0) * np.sqrt(d[lo:hi]))).astype(np.float32)
            a[lo:hi] = v
        out.append(a)
    return out
