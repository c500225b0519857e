"""Drop-in for the compiled `pointops_cuda` module (the reference's extensions/pointops): the two bound functions,
writing into the caller's tensors like the pybind originals (xyz (N,3) fp32, offsets (b,) int32, global indices)."""
from . import ops


def furthestsampling_cuda(b, n, xyz, offset, new_offset, tmp, idx):
    """idx (M,) int32 <- the samples of every segment; tmp (N,) fp32 holds the running minima (filled with 1e10 by
    the reference's caller).  b must equal the number of offsets."""
    if int(b) != offset.numel():
        raise RuntimeError("b=%d but offset holds %d segments" % (int(b), offset.numel()))
    ops.segment_fps_into(xyz, offset, new_offset, int(n), idx, tmp)


def knnquery_cuda(m, nsample, xyz, new_xyz, offset, new_offset, idx, dist2):
    """idx (m,nsample) int32, dist2 (m,nsample) fp32 (squared) <- the nsample nearest points of each query's segment."""
    if int(m) != new_xyz.size(0):
        raise RuntimeError("m=%d but new_xyz holds %d queries" % (int(m), new_xyz.size(0)))
    ops.segment_knn_into(nsample, xyz, new_xyz, offset, new_offset, idx, dist2)
