"""Approximate Earth Mover's Distance over variable-size clouds packed in one batch (csrc/segemd.cu).

Clouds are packed back to back, xyz1 (N, 3) and xyz2 (M, 3), with offset1 / offset2 (b,) int32 cumulative ends, the
layout of `pointops`.  Segment s of xyz1 is matched only against segment s of xyz2, with exactly the arithmetic of
emd.earth_mover_distance on that pair.  Nothing here reads the offsets on the host.

    segment_earth_mover_distance(xyz1, xyz2, offset1, offset2) -> (b,) cost per segment, differentiable in both clouds

A segment with an empty side costs 0 and its points get gradient 0.
"""
import torch

from . import ops


class SegmentEarthMoverDistanceFunction(torch.autograd.Function):
    """The forward keeps the per-level ratios (80 bytes per point), never the match; the backward rebuilds the match
    from them inside the kernels, as emd.EarthMoverDistanceFunction does."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, offset1, offset2):
        xyz1, xyz2 = xyz1.contiguous(), xyz2.contiguous()
        ratio_l, ratio_r = ops.segment_emd_match(xyz1, xyz2, offset1, offset2)
        cost = ops.segment_emd_cost(xyz1, xyz2, offset1, offset2, ratio_l, ratio_r)
        ctx.save_for_backward(xyz1, xyz2, offset1, offset2, ratio_l, ratio_r)
        return cost

    @staticmethod
    def backward(ctx, grad_cost):
        xyz1, xyz2, offset1, offset2, ratio_l, ratio_r = ctx.saved_tensors
        grad1, grad2 = ops.segment_emd_cost_grad(grad_cost.contiguous(), xyz1, xyz2, offset1, offset2, ratio_l, ratio_r)
        return grad1, grad2, None, None


def segment_earth_mover_distance(xyz1, xyz2, offset1, offset2):
    """xyz1 (N,3), xyz2 (M,3) fp32 CUDA, offset1 / offset2 (b,) int32 CUDA -> (b,) approximate EMD cost of each segment
    pair (no normalisation), differentiable in both clouds."""
    return SegmentEarthMoverDistanceFunction.apply(xyz1, xyz2, offset1, offset2)
