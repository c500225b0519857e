"""Chamfer distance over variable-size clouds packed in one batch (csrc/segchamfer.cu).

Clouds are packed back to back, xyz1 (N, 3) and xyz2 (M, 3), with offset1 / offset2 (b,) int32 cumulative ends, the
layout of `pointops`.  Segment s of xyz1 is matched only against segment s of xyz2; indices are global.  Nothing here
reads the offsets on the host.

    SegmentChamferFunction.apply(xyz1, xyz2, offset1, offset2) -> dist1, dist2, idx1, idx2
    SegmentChamferDistanceL2()(xyz1, xyz2, offset1, offset2)   -> mean over the clouds of mean(dist1) + mean(dist2)
    SegmentChamferDistanceL1()(xyz1, xyz2, offset1, offset2)   -> mean over the clouds of (mean(sqrt d1) + mean(sqrt d2)) / 2

Clouds with an empty side take no part in the losses; with none left the loss and its gradients are 0.
"""
import torch

from . import ops


class SegmentChamferFunction(torch.autograd.Function):
    """ops.segment_chamfer_forward with its gradient; idx1 / idx2 are not differentiable."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, offset1, offset2):
        dist1, dist2, idx1, idx2 = ops.segment_chamfer_forward(xyz1, xyz2, offset1, offset2)
        ctx.save_for_backward(xyz1, xyz2, idx1, idx2)
        ctx.mark_non_differentiable(idx1, idx2)
        return dist1, dist2, idx1, idx2

    @staticmethod
    def backward(ctx, grad_dist1, grad_dist2, *_):
        xyz1, xyz2, idx1, idx2 = ctx.saved_tensors
        gx1, gx2 = ops.segment_chamfer_backward(xyz1, xyz2, idx1, idx2, grad_dist1, grad_dist2)
        return gx1, gx2, None, None


class _SegmentChamferMeanLoss(torch.autograd.Function):
    """forward + cloud-weighted mean as one autograd node: the backward goes from the upstream scalar straight to the
    point gradients, as chamfer_dist._ChamferMeanLoss does for equal-size clouds."""

    @staticmethod
    def forward(ctx, xyz1, xyz2, offset1, offset2, l1):
        dist1, dist2, idx1, idx2 = ops.segment_chamfer_forward(xyz1, xyz2, offset1, offset2)
        state = torch.empty((4 * offset1.numel() + 1,), dtype=torch.int32, device=xyz1.device)
        loss3 = ops.segment_chamfer_loss(dist1, dist2, offset1, offset2, l1, state)
        ctx.save_for_backward(xyz1, xyz2, idx1, idx2, dist1, dist2, state)
        ctx.l1 = l1
        return loss3[0]

    @staticmethod
    def backward(ctx, grad_loss):
        xyz1, xyz2, idx1, idx2, dist1, dist2, state = ctx.saved_tensors
        gx1, gx2 = ops.segment_chamfer_loss_backward(xyz1, xyz2, idx1, idx2, dist1, dist2, state, grad_loss, ctx.l1)
        return gx1, gx2, None, None, None


class SegmentChamferDistanceL2(torch.nn.Module):
    """(1/|S|) sum over the clouds s of S of [mean_s dist1 + mean_s dist2]: ChamferDistanceL2 averaged over the clouds."""

    def forward(self, xyz1, xyz2, offset1, offset2):
        return _SegmentChamferMeanLoss.apply(xyz1, xyz2, offset1, offset2, False)


class SegmentChamferDistanceL1(torch.nn.Module):
    """(1/|S|) sum over S of [mean_s sqrt(dist1) + mean_s sqrt(dist2)] / 2: ChamferDistanceL1 averaged over the clouds."""

    def forward(self, xyz1, xyz2, offset1, offset2):
        return _SegmentChamferMeanLoss.apply(xyz1, xyz2, offset1, offset2, True)
