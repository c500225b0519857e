"""Approximate Earth Mover's Distance as an autograd Function that never holds the (B,m,n) match: the forward keeps
the per-level ratios (80 bytes per point) and the backward rebuilds the match from them inside the kernels."""
import torch

from . import ops


class EarthMoverDistanceFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xyz1, xyz2):
        xyz1, xyz2 = xyz1.contiguous(), xyz2.contiguous()
        ratio_l, ratio_r, _ = ops.emd_match(xyz1, xyz2)
        cost = ops.emd_cost(xyz1, xyz2, ratio_l=ratio_l, ratio_r=ratio_r)
        ctx.save_for_backward(xyz1, xyz2, ratio_l, ratio_r)
        return cost

    @staticmethod
    def backward(ctx, grad_cost):
        xyz1, xyz2, ratio_l, ratio_r = ctx.saved_tensors
        grad1, grad2 = ops.emd_cost_grad(grad_cost.contiguous(), xyz1, xyz2, ratio_l=ratio_l, ratio_r=ratio_r)
        return grad1, grad2


def earth_mover_distance(xyz1, xyz2):
    """xyz1 (B,n,3), xyz2 (B,m,3) fp32 CUDA -> (B,) approximate EMD cost (no normalisation), differentiable in both."""
    return EarthMoverDistanceFunction.apply(xyz1, xyz2)
