"""Sampling and kNN of variable-size clouds packed in one batch, with the reference's pointops interface:
xyz (N,3) fp32 holds the clouds back to back, offset / new_offset (b,) int32 the cumulative ends of the points and of
the samples / queries, and every returned index is global (a row of xyz)."""
import torch

from . import ops


def furthestsampling(xyz, offset, new_offset):
    """-> idx (new_offset[-1],) int32: furthest point sampling inside every segment, starting from its first point.
    Reads the largest segment size and the sample count on the host (one copy)."""
    return ops.segment_fps(xyz, offset, new_offset)


def knnquery(nsample, xyz, new_xyz, offset, new_offset):
    """-> (idx (M,nsample) int32, dist (M,nsample) fp32 Euclidean): the nsample nearest points of each query's own
    segment, ascending.  new_xyz=None queries the points themselves."""
    if new_xyz is None:
        new_xyz = xyz
    idx, dist2 = ops.segment_knn(nsample, xyz, new_xyz, offset, new_offset)
    return idx, torch.sqrt(dist2)
