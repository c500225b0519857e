"""Drop-in for the compiled `emd_cuda` module (the reference's extensions/emd): approxmatch_forward,
matchcost_forward and matchcost_backward with the reference's shapes (xyz (B,N,3) fp32, match (B,m,n) fp32)."""
from . import ops


def approxmatch_forward(xyz1, xyz2):
    """-> match (B,m,n)"""
    return ops.emd_match(xyz1, xyz2, materialize=True)[2]


def matchcost_forward(xyz1, xyz2, match):
    """-> cost (B,)"""
    return ops.emd_cost(xyz1, xyz2, match=match.contiguous())


def matchcost_backward(grad_cost, xyz1, xyz2, match):
    """-> [grad_xyz1 (B,n,3), grad_xyz2 (B,m,3)]"""
    return list(ops.emd_cost_grad(grad_cost.contiguous(), xyz1, xyz2, match=match.contiguous()))
