"""Torch-tensor host layer over the C ABI: allocates outputs, picks device / stream, raises on error.

PyTorch is plumbing here (device memory, streams, autograd glue); every computation is a
hand-written sm_100a kernel in csrc/.  No function in this module has a CPU or torch fallback:
a CPU tensor raises, a missing library raises.
"""
import threading

import torch

from . import _native


def _stream():
    return torch.cuda.current_stream().cuda_stream


class _NoGuard:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


_NO_GUARD = _NoGuard()


def _on(dev):
    """device guard for the launch: free when the tensor already lives on the current device (the
    torch.cuda.device context manager costs several microseconds per op otherwise)."""
    return _NO_GUARD if dev.index == torch.cuda.current_device() else torch.cuda.device(dev)


def _require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError("%s: CPU not supported" % name)  # sampling.cpp:36,84 of the reference


def _require_f32_contig(t, name):
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be a float tensor" % name)  # utils.h CHECK_IS_FLOAT
    if not t.is_contiguous():
        raise RuntimeError("%s must be a contiguous tensor" % name)  # utils.h CHECK_CONTIGUOUS


def _require_i32_contig(t, name):
    if t.dtype != torch.int32:
        raise RuntimeError("%s must be an int tensor" % name)  # utils.h CHECK_IS_INT
    if not t.is_contiguous():
        raise RuntimeError("%s must be a contiguous tensor" % name)


def _same_device(dev, **tensors):
    for name, t in tensors.items():
        if t is not None and t.device != dev:
            raise RuntimeError("%s is on %s, expected %s" % (name, t.device, dev))


def _dense_storage(t):
    """True when t's elements occupy exactly numel contiguous storage slots (any permutation)."""
    if t.numel() == 0 or t.is_contiguous():
        return True
    dims = sorted(((st, sz) for st, sz in zip(t.stride(), t.shape) if sz > 1))
    expect = 1
    for st, sz in dims:
        if st != expect:
            return False
        expect *= sz
    return True


# ------------------------------------------------------------------------------------------ FPS
def _deterministic():
    """torch.use_deterministic_algorithms(True) selects the gradients without float atomics (the *_det entry points)."""
    return torch.are_deterministic_algorithms_enabled()


def _workspace(nbytes, dev):
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=dev)


def fps_block_size(n):
    return int(_native.lib().pdae_fps_block_size(int(n)))


def furthest_point_sample(xyz, npoint):
    """pointnet2_utils.furthest_point_sample: xyz (B,N,3) f32 contiguous CUDA -> (B,npoint) int32."""
    _require_f32_contig(xyz, "xyz")
    _require_cuda(xyz, "furthest_point_sampling")
    if xyz.dim() != 3 or xyz.size(2) != 3:
        raise RuntimeError("xyz must have shape (B, N, 3)")
    b, n, _ = xyz.shape
    npoint = int(npoint)
    L = _native.lib()
    with _on(xyz.device):
        idx = torch.empty((b, npoint), dtype=torch.int32, device=xyz.device)
        nbytes = L.pdae_fps_workspace_bytes(b, n, npoint)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=xyz.device) if nbytes else None
        rc = L.pdae_fps_f32(xyz.data_ptr(), b, n, npoint, idx.data_ptr(), ws.data_ptr() if nbytes else None, nbytes,
                            _stream())
    _native.check(rc, "pdae_fps_f32")
    return idx


def fps_gather(data, number):
    """Fused utils/misc.py:13-20 `fps`: data (B,N,C>=3) -> (fps_idx (B,G) int32, fps_data (B,G,C))."""
    _require_cuda(data, "fps")
    if data.dim() != 3 or data.size(2) < 3:
        raise RuntimeError("data must have shape (B, N, C>=3)")
    src = data.detach()
    if src.dtype != torch.float32 or not src.is_contiguous():
        src = src.float().contiguous()
    b, n, c = src.shape
    number = int(number)
    L = _native.lib()
    with _on(src.device):
        idx = torch.empty((b, number), dtype=torch.int32, device=src.device)
        centers = torch.empty((b, number, c), dtype=torch.float32, device=src.device)
        nbytes = L.pdae_fps_workspace_bytes(b, n, number)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=src.device) if nbytes else None
        rc = L.pdae_fps_gather_f32(src.data_ptr(), b, n, c, number, idx.data_ptr(), centers.data_ptr(),
                                   ws.data_ptr() if nbytes else None, nbytes, _stream())
    _native.check(rc, "pdae_fps_gather_f32")
    return idx, centers


# --------------------------------------------------------------------------------------- gather
def gather_points(features, idx):
    _require_f32_contig(features, "features")
    _require_i32_contig(idx, "idx")
    _require_cuda(features, "gather_points")
    _require_cuda(idx, "gather_points")
    b, c, n = features.shape
    m = idx.size(1)
    if idx.size(0) != b:
        raise RuntimeError("features and idx disagree on the batch size")
    with _on(features.device):
        out = torch.empty((b, c, m), dtype=torch.float32, device=features.device)
        rc = _native.lib().pdae_gather_f32(features.data_ptr(), idx.data_ptr(), b, c, n, m, out.data_ptr(), _stream())
    _native.check(rc, "pdae_gather_f32")
    return out


def gather_points_grad(grad_out, idx, n):
    _require_f32_contig(grad_out, "grad_out")
    _require_i32_contig(idx, "idx")
    _require_cuda(grad_out, "gather_points_grad")
    _require_cuda(idx, "gather_points_grad")
    b, c, m = grad_out.shape
    with _on(grad_out.device):
        out = torch.empty((b, c, int(n)), dtype=torch.float32, device=grad_out.device)
        L = _native.lib()
        if _deterministic():
            nbytes = L.pdae_gather_grad_det_workspace_bytes(b, int(n), m)
            ws = _workspace(nbytes, grad_out.device)
            rc = L.pdae_gather_grad_det_f32(grad_out.data_ptr(), idx.data_ptr(), b, c, int(n), m, out.data_ptr(), ws.data_ptr(),
                                            nbytes, _stream())
        else:
            rc = L.pdae_gather_grad_f32(grad_out.data_ptr(), idx.data_ptr(), b, c, int(n), m, out.data_ptr(), _stream())
    _native.check(rc, "pdae_gather_grad_f32")
    return out


# ------------------------------------------------------------------------------------------ kNN
def _knn_workspace(b, r, q, d, k, dev):
    """Scratch for the chunked form of scene-scale searches (few queries, long reference cloud); None for every other
    shape.  Comes from the caching allocator on the current stream, like every other workspace."""
    nbytes = int(_native.lib().pdae_knn_workspace_bytes(b, r, q, d, k))
    if nbytes <= 0:
        return None, 0
    return torch.empty(nbytes, dtype=torch.uint8, device=dev), nbytes


def knn_points(ref, query, k, out_kq=False, want_dist=True):
    """ref (B,R,D), query (B,Q,D) f32 contiguous -> (dist (B,Q,k)|(B,k,Q) f32 or None, idx int64)."""
    _require_cuda(ref, "knn")
    _require_cuda(query, "knn")
    _require_f32_contig(ref, "ref")      # raw pointers go to the kernel: no silent reinterpretation of strides / dtypes
    _require_f32_contig(query, "query")
    if query.device != ref.device:
        raise RuntimeError("ref is on %s but query is on %s" % (ref.device, query.device))
    b, r, d = ref.shape
    q = query.size(1)
    k = int(k)
    if query.size(0) != b or query.size(2) != d:
        raise RuntimeError("ref.shape=%s != query.shape=%s" % (tuple(ref.shape), tuple(query.shape)))
    if not (1 <= k <= r):
        raise RuntimeError("k=%d must satisfy 1 <= k <= %d reference points" % (k, r))
    shape = (b, k, q) if out_kq else (b, q, k)
    with _on(ref.device):
        idx = torch.empty(shape, dtype=torch.int64, device=ref.device)
        dist = torch.empty(shape, dtype=torch.float32, device=ref.device) if want_dist else None
        ws, ws_bytes = _knn_workspace(b, r, q, d, k, ref.device)
        rc = _native.lib().pdae_knn_ws_f32(ref.data_ptr(), query.data_ptr(), b, r, q, d, k, 1 if out_kq else 0,
                                           dist.data_ptr() if want_dist else None, idx.data_ptr(),
                                           ws.data_ptr() if ws is not None else None, ws_bytes, _stream())
    _native.check(rc, "pdae_knn_ws_f32")
    return dist, idx


def knn_keys(ref_local, query, k, ref_offset):
    """This rank's k best candidates per query from its slice of the reference cloud (global index of the slice's first
    point = ref_offset): int64 (B,Q,k), ascending packed (squared-distance bits << 32 | global index) keys."""
    _require_cuda(ref_local, "knn_keys")
    _require_cuda(query, "knn_keys")
    _require_f32_contig(ref_local, "ref_local")
    _require_f32_contig(query, "query")
    b, r, d = ref_local.shape
    q = query.size(1)
    if query.size(0) != b or query.size(2) != d:
        raise RuntimeError("ref.shape=%s != query.shape=%s" % (tuple(ref_local.shape), tuple(query.shape)))
    with _on(query.device):
        keys = torch.empty((b, q, int(k)), dtype=torch.int64, device=query.device)
        rc = _native.lib().pdae_knn_keys_u64(ref_local.data_ptr(), query.data_ptr(), b, r, q, d, int(k), int(ref_offset),
                                             keys.data_ptr(), _stream())
    _native.check(rc, "pdae_knn_keys_u64")
    return keys


def knn_merge_keys(keys_all, out_kq=False, want_dist=True):
    """keys_all int64 (W,B,Q,k): the all-gathered per-rank candidate lists -> (dist, idx) exactly as knn_points on the
    whole reference cloud."""
    _require_cuda(keys_all, "knn_merge_keys")
    if keys_all.dtype != torch.int64 or keys_all.dim() != 4 or not keys_all.is_contiguous():
        raise RuntimeError("keys_all must be a contiguous int64 tensor of shape (W, B, Q, k)")
    w, b, q, k = keys_all.shape
    shape = (b, k, q) if out_kq else (b, q, k)
    with _on(keys_all.device):
        idx = torch.empty(shape, dtype=torch.int64, device=keys_all.device)
        dist = torch.empty(shape, dtype=torch.float32, device=keys_all.device) if want_dist else None
        rc = _native.lib().pdae_knn_merge_keys_u64(keys_all.data_ptr(), w, b, q, k, 1 if out_kq else 0,
                                                   dist.data_ptr() if want_dist else None, idx.data_ptr(), _stream())
    _native.check(rc, "pdae_knn_merge_keys_u64")
    return dist, idx


def group_points_knn(xyz, center, group_size, want_idx=True, subtract_center=True):
    """Fused Group tail: xyz (B,N,3), center (B,G,3) -> (neighborhood (B,G,M,3), idx (B,G,M) int64|None).
    subtract_center=False returns the neighbours themselves (xyz[idx]), the gather of dropout_patch_random."""
    _require_cuda(xyz, "group")
    _require_f32_contig(xyz, "xyz")
    _require_f32_contig(center, "center")
    b, n, _ = xyz.shape
    g = center.size(1)
    m = int(group_size)
    if not (1 <= m <= n):
        raise RuntimeError("group_size=%d must satisfy 1 <= group_size <= %d points" % (m, n))
    with _on(xyz.device):
        nb = torch.empty((b, g, m, 3), dtype=torch.float32, device=xyz.device)
        idx = torch.empty((b, g, m), dtype=torch.int64, device=xyz.device) if want_idx else None
        if subtract_center:
            ws, ws_bytes = _knn_workspace(b, n, g, 3, m, xyz.device)
            rc = _native.lib().pdae_group_ws_f32(xyz.data_ptr(), center.data_ptr(), b, n, g, m,
                                                 idx.data_ptr() if want_idx else None, nb.data_ptr(),
                                                 ws.data_ptr() if ws is not None else None, ws_bytes, _stream())
        else:
            rc = _native.lib().pdae_group_gather_f32(xyz.data_ptr(), center.data_ptr(), b, n, g, m,
                                                     idx.data_ptr() if want_idx else None, nb.data_ptr(), _stream())
    _native.check(rc, "pdae_group_f32")
    return nb, idx


def fps_group(xyz, num_group, group_size, want_idx=False, overlap_previous=False):
    """The whole patchifier of `Group.forward` (models/PointCAE_transformer.py:61-86) in one call / one launch:
    xyz (B,N,3) -> (fps_idx (B,G) int32, center (B,G,3), neighborhood (B,G,M,3) centre-subtracted, idx (B,G,M) int64|None).
    Bit-identical with fps_gather + group_points_knn (the form shapes outside 512..2048 points / M <= 32 still take).
    overlap_previous=True: the caller vouches that the kernel queued before this call on the current stream does not
    produce `xyz` (the Chamfer forward of the same step); the launch then uses programmatic stream serialization and its
    CTAs start as that kernel's CTAs exit instead of after its whole grid has drained."""
    _require_cuda(xyz, "fps_group")
    _require_f32_contig(xyz, "xyz")
    if xyz.dim() != 3 or xyz.size(2) != 3:
        raise RuntimeError("xyz must have shape (B, N, 3)")
    b, n, _ = xyz.shape
    g, m = int(num_group), int(group_size)
    if n < 1 or not (1 <= m <= n):
        raise RuntimeError("group_size=%d must satisfy 1 <= group_size <= %d points" % (m, n))
    L = _native.lib()
    with _on(xyz.device):
        fps_idx = torch.empty((b, g), dtype=torch.int32, device=xyz.device)
        center = torch.empty((b, g, 3), dtype=torch.float32, device=xyz.device)
        nb = torch.empty((b, g, m, 3), dtype=torch.float32, device=xyz.device)
        idx = torch.empty((b, g, m), dtype=torch.int64, device=xyz.device) if want_idx else None
        nbytes = int(L.pdae_fps_group_workspace_bytes(b, n, g, m))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=xyz.device) if nbytes else None
        rc = L.pdae_fps_group_ex_f32(xyz.data_ptr(), b, n, g, m, fps_idx.data_ptr(), center.data_ptr(),
                                     idx.data_ptr() if want_idx else None, nb.data_ptr(),
                                     ws.data_ptr() if nbytes else None, nbytes, 1 if overlap_previous else 0, _stream())
    _native.check(rc, "pdae_fps_group_ex_f32")
    return fps_idx, center, nb, idx


class StepBuffers:
    """Outputs and workspace of `hot_step`, allocated once per shape (a training loop reuses them every step).
    deterministic (default: torch.are_deterministic_algorithms_enabled()) sizes the workspace for the deterministic
    backward as well; `hot_step` grows it in place when a step needs it and the buffers were built without it."""

    def __init__(self, b, n, g, m, device, deterministic=None):
        if deterministic is None:
            deterministic = _deterministic()
        self.shape = (b, n, g, m)
        f32, i32 = torch.float32, torch.int32
        with _on(device):
            self.fps_idx = torch.empty((b, g), dtype=i32, device=device)
            self.center = torch.empty((b, g, 3), dtype=f32, device=device)
            self.neighborhood = torch.empty((b, g, m, 3), dtype=f32, device=device)
            self.dist1 = torch.empty((b, n), dtype=f32, device=device)
            self.dist2 = torch.empty((b, n), dtype=f32, device=device)
            self.idx1 = torch.empty((b, n), dtype=i32, device=device)
            self.idx2 = torch.empty((b, n), dtype=i32, device=device)
            self.loss3 = torch.empty(3, dtype=f32, device=device)
            self.gpred = torch.empty((b, n, 3), dtype=f32, device=device)
            self.gcloud = torch.empty((b, n, 3), dtype=f32, device=device)
            self.flags = 0
            self.ws_bytes = 0
            self.ws = None
            self.reserve(deterministic)

    def reserve(self, deterministic):
        """make the workspace large enough for the deterministic (or default) step; only `ws` changes, the outputs stay"""
        flags = 1 if deterministic else 0  # PDAE_STEP_DETERMINISTIC
        if self.ws is not None and flags <= self.flags:
            return
        device = self.loss3.device
        with _on(device):
            nbytes = int(_native.lib().pdae_step_ex_workspace_bytes(*self.shape, flags))
            self.ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        self.ws_bytes, self.flags = nbytes, flags


def hot_step(cloud, pred, num_group, group_size, gloss, buffers=None, deterministic=None):
    """One step of the hot path in ONE native call (csrc/step.cu): Chamfer forward of `pred` against `cloud`, the patchifier
    of `cloud` as a programmatic dependent launch, the fused mean loss and the gradients of that loss scaled by the device
    scalar `gloss`, on the current stream + two library-owned helper streams.  -> StepBuffers (neighborhood, center,
    fps_idx, dist1/2, idx1/2, loss3 = [loss, mean1, mean2], gpred, gcloud); the values of fps_group + chamfer_forward +
    chamfer_mean_loss + chamfer_loss_backward bit for bit.  deterministic (default: torch.are_deterministic_algorithms_enabled())
    selects the backward without float atomics, as chamfer_loss_backward does under that flag."""
    _require_cuda(cloud, "hot_step")
    _require_f32_contig(cloud, "cloud")
    _require_f32_contig(pred, "pred")
    _same_device(cloud.device, pred=pred, gloss=gloss)
    if cloud.dim() != 3 or cloud.size(2) != 3 or pred.shape != cloud.shape:
        raise RuntimeError("cloud and pred must both have shape (B, N, 3)")
    b, n, _ = cloud.shape
    g, m = int(num_group), int(group_size)
    if n < 1 or not (1 <= m <= n):
        raise RuntimeError("group_size=%d must satisfy 1 <= group_size <= %d points" % (m, n))
    det = _deterministic() if deterministic is None else bool(deterministic)
    if buffers is None or buffers.shape != (b, n, g, m) or buffers.loss3.device != cloud.device:
        buffers = StepBuffers(b, n, g, m, cloud.device, deterministic=det)
    buffers.reserve(det)  # the caller's outputs are kept: only a too-small workspace is replaced
    o = buffers
    with _on(cloud.device):
        args = (cloud.data_ptr(), pred.data_ptr(), b, n, g, m, o.fps_idx.data_ptr(), o.center.data_ptr(), o.neighborhood.data_ptr(),
                o.dist1.data_ptr(), o.dist2.data_ptr(), o.idx1.data_ptr(), o.idx2.data_ptr(), o.loss3.data_ptr(), gloss.data_ptr(),
                o.gpred.data_ptr(), o.gcloud.data_ptr(), o.ws.data_ptr(), o.ws_bytes)
        if det:
            rc = _native.lib().pdae_step_ex_f32(*args, 1, _stream())  # PDAE_STEP_DETERMINISTIC
        else:
            rc = _native.lib().pdae_step_f32(*args, _stream())
    _native.check(rc, "pdae_step_f32")
    return o


# -------------------------------------------------------------------- affine corruptions (SURVEY.md 8f row 3)
def _affine_mats(mats, b, dev):
    """(B,T,3,3) matrices, any device -> contiguous fp32 on `dev` (one small H2D copy when they come from the host,
    where the reference builds them too)."""
    if mats.dim() != 4 or mats.size(0) != b or tuple(mats.shape[2:]) != (3, 3):
        raise RuntimeError("mats must have shape (B, T, 3, 3) with B = %d" % b)
    return mats.to(device=dev, dtype=torch.float32).contiguous()


def _affine_launch(points, center, mats):
    b, t = mats.size(0), mats.size(1)
    p = points.numel() // (3 * b) if b else 0
    g = center.numel() // (3 * b) if b else 0
    with _on(points.device):
        out_p, out_c = torch.empty_like(points), torch.empty_like(center)
        rc = _native.lib().pdae_affine_points_f32(points.data_ptr(), center.data_ptr(), mats.data_ptr(), b, p, g, t,
                                                  out_p.data_ptr(), out_c.data_ptr(), _stream())
    _native.check(rc, "pdae_affine_points_f32")
    return out_p, out_c


class _AffinePoints(torch.autograd.Function):
    """y = x @ R_0 @ ... @ R_{T-1} per cloud; grad_x = grad_y @ R_{T-1}^T @ ... @ R_0^T (same kernel)."""

    @staticmethod
    def forward(ctx, points, center, mats):
        ctx.save_for_backward(mats)
        return _affine_launch(points, center, mats)

    @staticmethod
    def backward(ctx, gp, gc):
        (mats,) = ctx.saved_tensors
        back = mats.flip(1).transpose(2, 3).contiguous()
        gp, gc = _affine_launch(gp.contiguous(), gc.contiguous(), back)
        return gp, gc, None


def affine_points(points, center, mats):
    """One-launch `corrupt_data` (datasets/corrupt_util_tensor.py:706-728): points (B,...,3) and center (B,G,3) fp32
    CUDA, mats (B,T,3,3) applied in order to row vectors -> (points', center') with the input shapes."""
    _require_cuda(points, "corrupt_data")
    _require_cuda(center, "corrupt_data")
    if points.size(-1) != 3 or center.size(-1) != 3 or points.size(0) != center.size(0):
        raise RuntimeError("points (B,...,3) and center (B,G,3) expected")
    if mats.size(1) > 8:
        raise RuntimeError("at most 8 chained matrices")
    pts = points if points.dtype == torch.float32 and points.is_contiguous() else points.float().contiguous()
    ctr = center if center.dtype == torch.float32 and center.is_contiguous() else center.float().contiguous()
    mats = _affine_mats(mats, points.size(0), points.device)
    if pts.requires_grad or ctr.requires_grad:
        return _AffinePoints.apply(pts, ctr, mats)
    return _affine_launch(pts, ctr, mats)


def group_affine(xyz, center, group_size, mats, want_idx=False):
    """Fused Group tail + corrupt_data + re-centring (models/PointCAE_transformer.py:1010-1017):
    xyz (B,N,3), center (B,G,3), mats (B,T,3,3) -> neighborhood (B,G,M,3) [= ((x-c)+c)-c], t_neighborhood (B,G,M,3),
    t_center (B,G,3), idx (B,G,M) int64 | None.  No gradient (the patchifier has none in the reference either)."""
    _require_cuda(xyz, "group")
    _require_f32_contig(xyz, "xyz")
    _require_f32_contig(center, "center")
    b, n, _ = xyz.shape
    g = center.size(1)
    m = int(group_size)
    if not (1 <= m <= n):
        raise RuntimeError("group_size=%d must satisfy 1 <= group_size <= %d points" % (m, n))
    if mats.size(1) > 8:
        raise RuntimeError("at most 8 chained matrices")
    mats = _affine_mats(mats, b, xyz.device)
    with _on(xyz.device):
        nb = torch.empty((b, g, m, 3), dtype=torch.float32, device=xyz.device)
        tnb = torch.empty_like(nb)
        tc = torch.empty((b, g, 3), dtype=torch.float32, device=xyz.device)
        idx = torch.empty((b, g, m), dtype=torch.int64, device=xyz.device) if want_idx else None
        rc = _native.lib().pdae_group_affine_f32(xyz.data_ptr(), center.data_ptr(), mats.data_ptr(), b, n, g, m, mats.size(1),
                                                 idx.data_ptr() if want_idx else None, nb.data_ptr(), tnb.data_ptr(),
                                                 tc.data_ptr(), _stream())
    _native.check(rc, "pdae_group_affine_f32")
    return nb, tnb, tc, idx


def fps_group_affine(xyz, num_group, group_size, mats, want_idx=False):
    """FPS + centre gather + `group_affine` in one call (one launch for batches of >= 48 clouds of 512..2048 points):
    xyz (B,N,3), mats (B,T,3,3) -> (fps_idx, center, neighborhood, t_neighborhood, t_center, idx|None); the values of
    fps_gather followed by group_affine bit for bit."""
    _require_cuda(xyz, "fps_group_affine")
    _require_f32_contig(xyz, "xyz")
    if xyz.dim() != 3 or xyz.size(2) != 3:
        raise RuntimeError("xyz must have shape (B, N, 3)")
    b, n, _ = xyz.shape
    g, m = int(num_group), int(group_size)
    if n < 1 or not (1 <= m <= n):
        raise RuntimeError("group_size=%d must satisfy 1 <= group_size <= %d points" % (m, n))
    if mats.size(1) > 8:
        raise RuntimeError("at most 8 chained matrices")
    mats = _affine_mats(mats, b, xyz.device)
    L = _native.lib()
    with _on(xyz.device):
        fps_idx = torch.empty((b, g), dtype=torch.int32, device=xyz.device)
        center = torch.empty((b, g, 3), dtype=torch.float32, device=xyz.device)
        nb = torch.empty((b, g, m, 3), dtype=torch.float32, device=xyz.device)
        tnb = torch.empty_like(nb)
        tc = torch.empty_like(center)
        idx = torch.empty((b, g, m), dtype=torch.int64, device=xyz.device) if want_idx else None
        nbytes = int(L.pdae_fps_group_workspace_bytes(b, n, g, m))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=xyz.device) if nbytes else None
        rc = L.pdae_fps_group_affine_f32(xyz.data_ptr(), mats.data_ptr(), b, n, g, m, mats.size(1), fps_idx.data_ptr(),
                                         center.data_ptr(), idx.data_ptr() if want_idx else None, nb.data_ptr(),
                                         tnb.data_ptr(), tc.data_ptr(), ws.data_ptr() if nbytes else None, nbytes, _stream())
    _native.check(rc, "pdae_fps_group_affine_f32")
    return fps_idx, center, nb, tnb, tc, idx


# -------------------------------------------------------------------------------------- Chamfer
_scan_events = threading.local()


class chamfer_scan_event:
    """`with ops.chamfer_scan_event(ev): loss = ChamferDistanceL2()(a, b)` -- the next chamfer_forward on this thread
    records the torch.cuda.Event `ev` on its stream right after the FMA-bound scan kernel (before the latency-bound
    column recovery).  Work on another stream that should overlap the tail of the step instead of the scan -- the
    patchifier's kNN in bench.py -- waits on it (`Group.forward(xyz, knn_after=ev)`).  Scheduling only: results are
    unchanged."""

    def __init__(self, event):
        self.event = event

    def __enter__(self):
        _scan_events.pending = self.event
        return self.event

    def __exit__(self, *a):
        _scan_events.pending = None
        return False


class chamfer_column_split:
    """`with ops.chamfer_column_split(False): ...` -- forwards issued by this thread inside the block get a workspace
    for the column keys only, so the library runs every row block against the whole reference cloud in one CTA.
    The split (default: automatic, see pdae_chamfer_fwd_workspace_bytes) shortens a forward that has the GPU to
    itself by evening out the SMs' load (128 x 2048^2: 178 -> 168 us; 1 x 100k^2: 3.6 -> 2.4 ms); a caller that
    overlaps other kernels with the forward on a second stream (bench.py's patchifier branch) already fills the idle
    tail with them and is better off without the split's extra prologues (step 232 vs 239 us).  Scheduling only:
    results are identical."""

    def __init__(self, enabled):
        self.enabled = bool(enabled)

    def __enter__(self):
        self.prev = getattr(_scan_events, "split", True)
        _scan_events.split = self.enabled
        return self

    def __exit__(self, *a):
        _scan_events.split = self.prev
        return False


def chamfer_forward(xyz1, xyz2, symmetric=True, scan_done=None):
    """chamfer.forward: returns [dist1 (B,N), dist2 (B,M), idx1 int32, idx2 int32].
    scan_done: optional torch.cuda.Event recorded between the scan and the column recovery (see chamfer_scan_event).

    Reference-faithful storage semantics (chamfer.cu:159-164 reads raw data_ptr): a tensor whose
    elements densely fill their storage is read in *storage order* as [B][size(1)][3], even when it
    is a transposed view -- exactly what the reference computes for
    models/PointCAE_transformer.py:1059-1066.  Anything else (gaps, overlaps, wrong dtype) raises
    instead of reading out of bounds like the reference would.
    """
    for t, name in ((xyz1, "xyz1"), (xyz2, "xyz2")):
        _require_cuda(t, "chamfer.forward")
        if t.dtype != torch.float32:
            raise RuntimeError("%s must be a float tensor" % name)
        if t.dim() != 3 or t.size(2) < 3:
            raise RuntimeError("%s must have shape (B, N, 3)" % name)
        if not _dense_storage(t):
            raise RuntimeError("%s must densely fill its storage (the reference reads raw memory)" % name)
        # size(2) > 3 (ChamferDistanceL2_withnormal_normalindex hands in (B,N,6), __init__.py:302-304): the
        # reference still walks the storage as [B][size(1)][3]; that stays inside the allocation, so it is kept.
    b, n, _ = xyz1.shape
    m = xyz2.size(1)
    if xyz2.size(0) != b:
        raise RuntimeError("batch sizes differ: %d vs %d" % (b, xyz2.size(0)))
    dev = xyz1.device
    _same_device(dev, xyz2=xyz2)
    with _on(dev):
        dist1 = torch.empty((b, n), dtype=torch.float32, device=dev)
        dist2 = torch.empty((b, m), dtype=torch.float32, device=dev)
        idx1 = torch.empty((b, n), dtype=torch.int32, device=dev)
        idx2 = torch.empty((b, m), dtype=torch.int32, device=dev)
        L = _native.lib()
        # with the workspace every pair is evaluated once for both directions; without it (symmetric=False)
        # each direction is scanned separately -- same results, twice the arithmetic
        nbytes = L.pdae_chamfer_fwd_workspace_bytes(b, n, m) if symmetric else 0
        if nbytes and not getattr(_scan_events, "split", True):
            nbytes = b * min(n, m) * 8  # column keys only: no column split (see chamfer_column_split)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev) if nbytes else None
        args = (xyz1.data_ptr(), xyz2.data_ptr(), b, n, m, dist1.data_ptr(), dist2.data_ptr(), idx1.data_ptr(),
                idx2.data_ptr(), ws.data_ptr() if nbytes else None, nbytes)
        if scan_done is None:
            scan_done = getattr(_scan_events, "pending", None)
            _scan_events.pending = None  # one-shot: only the first forward inside the context records
        if scan_done is None:
            rc = L.pdae_chamfer_fwd_f32(*args, _stream())
        else:
            rc = L.pdae_chamfer_fwd_phase_f32(*args, 1, _stream())
            _native.check(rc, "pdae_chamfer_fwd_phase_f32")
            scan_done.record(torch.cuda.current_stream())
            rc = L.pdae_chamfer_fwd_phase_f32(*args, 2, _stream())
    _native.check(rc, "pdae_chamfer_fwd_f32")
    return [dist1, dist2, idx1, idx2]


def chamfer_backward(xyz1, xyz2, idx1, idx2, grad_dist1, grad_dist2):
    """chamfer.backward: returns [grad_xyz1, grad_xyz2], allocated like the reference's
    zeros_like (strides of the inputs preserved, chamfer.cu:212-213) and written in storage order."""
    b, n, _ = xyz1.shape
    m = xyz2.size(1)
    dev = xyz1.device
    for t, name in ((xyz1, "xyz1"), (xyz2, "xyz2")):
        _require_cuda(t, "chamfer.backward")
        if t.dtype != torch.float32 or not _dense_storage(t):
            raise RuntimeError("%s must be a float tensor that densely fills its storage" % name)
    if idx1.dtype != torch.int32 or idx2.dtype != torch.int32:
        raise RuntimeError("idx1 / idx2 must be the int tensors returned by chamfer.forward")
    _same_device(dev, xyz2=xyz2, idx1=idx1, idx2=idx2, grad_dist1=grad_dist1, grad_dist2=grad_dist2)
    idx1, idx2 = idx1.contiguous(), idx2.contiguous()
    if tuple(idx1.shape) != (b, n) or tuple(idx2.shape) != (b, m):
        raise RuntimeError("idx1 / idx2 do not match the clouds' shapes")
    grad_dist1 = grad_dist1.contiguous().float()
    grad_dist2 = grad_dist2.contiguous().float()
    with _on(dev):
        # preserve_format: dense inputs keep their strides; wider-than-3 rows are only partly written -> zeros
        gx1 = torch.empty_like(xyz1) if xyz1.size(2) == 3 else torch.zeros_like(xyz1)
        gx2 = torch.empty_like(xyz2) if xyz2.size(2) == 3 else torch.zeros_like(xyz2)
        L = _native.lib()
        args = (xyz1.data_ptr(), xyz2.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), grad_dist1.data_ptr(),
                grad_dist2.data_ptr(), b, n, m, gx1.data_ptr(), gx2.data_ptr())
        if _deterministic():
            nbytes = L.pdae_chamfer_bwd_det_workspace_bytes(b, n, m)
            ws = _workspace(nbytes, dev)
            rc = L.pdae_chamfer_bwd_det_f32(*args, ws.data_ptr(), nbytes, _stream())
        else:
            rc = L.pdae_chamfer_bwd_f32(*args, _stream())
    _native.check(rc, "pdae_chamfer_bwd_f32")
    return [gx1, gx2]


def chamfer_mean_loss(dist1, dist2, l1=False):
    """Fused loss epilogue: -> float32 tensor (3,) = [loss, mean term 1, mean term 2] with
    loss = mean(dist1) + mean(dist2) (L2, extensions/chamfer_dist/__init__.py:43) or
    (mean(sqrt(dist1)) + mean(sqrt(dist2))) / 2 (L1, :413-417).  Two launches, deterministic."""
    for t in (dist1, dist2):
        _require_cuda(t, "chamfer_mean_loss")
        _require_f32_contig(t, "dist")
    b, n = dist1.shape
    m = dist2.size(1)
    dev = dist1.device
    L = _native.lib()
    with _on(dev):
        out = torch.empty(3, dtype=torch.float32, device=dev)
        nbytes = L.pdae_chamfer_loss_workspace_bytes()
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        rc = L.pdae_chamfer_loss_f32(dist1.data_ptr(), dist2.data_ptr(), b, n, m, 1 if l1 else 0, out.data_ptr(),
                                     ws.data_ptr(), nbytes, _stream())
    _native.check(rc, "pdae_chamfer_loss_f32")
    return out


def chamfer_loss_backward(xyz1, xyz2, idx1, idx2, dist1, dist2, grad_loss, w1, w2, l1=False):
    """Gradients of w1*mean(f(dist1)) + w2*mean(f(dist2)) (f = identity, or sqrt when l1) times the device scalar
    grad_loss, straight from the saved argmin -- what autograd reaches through MeanBackward (+SqrtBackward) and
    chamfer.backward in the reference.  Same stride rules as chamfer_backward."""
    b, n, _ = xyz1.shape
    m = xyz2.size(1)
    dev = xyz1.device
    for t, name in ((xyz1, "xyz1"), (xyz2, "xyz2")):
        _require_cuda(t, "chamfer_loss_backward")
        if t.dtype != torch.float32 or not _dense_storage(t):
            raise RuntimeError("%s must be a float tensor that densely fills its storage" % name)
    if idx1.dtype != torch.int32 or idx2.dtype != torch.int32:
        raise RuntimeError("idx1 / idx2 must be the int tensors returned by chamfer.forward")
    _same_device(dev, xyz2=xyz2, idx1=idx1, idx2=idx2, dist1=dist1, dist2=dist2, grad_loss=grad_loss)
    grad_loss = grad_loss.reshape(-1)
    if grad_loss.numel() != 1 or not grad_loss.is_cuda:
        raise RuntimeError("grad_loss must be a one-element CUDA tensor")
    grad_loss = grad_loss.float().contiguous()
    with _on(dev):
        gx1 = torch.empty_like(xyz1) if xyz1.size(2) == 3 else torch.zeros_like(xyz1)
        gx2 = torch.empty_like(xyz2) if xyz2.size(2) == 3 else torch.zeros_like(xyz2)
        idx1, idx2, dist1, dist2 = idx1.contiguous(), idx2.contiguous(), dist1.contiguous(), dist2.contiguous()
        L = _native.lib()
        args = (xyz1.data_ptr(), xyz2.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), dist1.data_ptr(), dist2.data_ptr(),
                grad_loss.data_ptr(), float(w1), float(w2), b, n, m, 1 if l1 else 0, gx1.data_ptr(), gx2.data_ptr())
        if _deterministic():
            nbytes = L.pdae_chamfer_bwd_det_workspace_bytes(b, n, m)
            ws = _workspace(nbytes, dev)
            rc = L.pdae_chamfer_loss_bwd_det_f32(*args, ws.data_ptr(), nbytes, _stream())
        else:
            rc = L.pdae_chamfer_loss_bwd_f32(*args, _stream())
    _native.check(rc, "pdae_chamfer_loss_bwd_f32")
    return [gx1, gx2]


PAIR_METRICS = {"dis_l2": 0, "dis_normalized_l2": 1, "dis_normalized_l1": 2, "dis_normalized_l2_strict": 3}


class MatchedPairLoss(torch.autograd.Function):
    """mean_j metric(a_j, b[idx1[j]]) + mean_j metric(b_j, a[idx2[j]]) over the Chamfer match (one forward launch, two
    backward launches; csrc/pairloss.cu) -- the normal / curvature / position terms of ChamferDistanceL2_withnormal*
    (extensions/chamfer_dist/__init__.py:143-165) without their gather / normalize / difference / mean chains."""

    @staticmethod
    def forward(ctx, a, b, idx1, idx2, metric):
        a, b = a.contiguous(), b.contiguous()
        idx1, idx2 = idx1.contiguous(), idx2.contiguous()
        bs, n, d = a.shape
        m = b.size(1)
        L = _native.lib()
        with _on(a.device):
            partial = torch.empty((int(L.pdae_pair_loss_partial_count(bs, n, m)), 2), dtype=torch.float64, device=a.device)
            rc = L.pdae_pair_loss_fwd_f64(a.data_ptr(), b.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), bs, n, m, d, int(metric),
                                          partial.data_ptr(), _stream())
        _native.check(rc, "pdae_pair_loss_fwd_f64")
        sums = partial.sum(dim=0)
        ctx.save_for_backward(a, b, idx1, idx2)
        ctx.metric = int(metric)
        return (sums[0] / (bs * n) + sums[1] / (bs * m)).float()

    @staticmethod
    def backward(ctx, g):
        a, b, idx1, idx2 = ctx.saved_tensors
        bs, n, d = a.shape
        m = b.size(1)
        with _on(a.device):
            ga, gb = torch.empty_like(a), torch.empty_like(b)
            gl = g.reshape(1).float().contiguous()
            L = _native.lib()
            args = (a.data_ptr(), b.data_ptr(), idx1.data_ptr(), idx2.data_ptr(), gl.data_ptr(), 1.0 / (bs * n), 1.0 / (bs * m),
                    bs, n, m, d, ctx.metric, ga.data_ptr(), gb.data_ptr())
            if _deterministic():
                nbytes = L.pdae_pair_loss_bwd_det_workspace_bytes(bs, n, m)
                ws = _workspace(nbytes, a.device)
                rc = L.pdae_pair_loss_bwd_det_f32(*args, ws.data_ptr(), nbytes, _stream())
            else:
                rc = L.pdae_pair_loss_bwd_f32(*args, _stream())
        _native.check(rc, "pdae_pair_loss_bwd_f32")
        return ga, gb, None, None, None


def matched_pair_loss(a, b, idx1, idx2, metric):
    """fused form when it applies (CUDA fp32, <= 8 attribute channels, int32 match indices), else None"""
    code = PAIR_METRICS.get(metric)
    if (code is None or not a.is_cuda or a.dtype != torch.float32 or b.dtype != torch.float32 or a.dim() != 3 or b.dim() != 3
            or a.size(2) != b.size(2) or a.size(2) > 8 or idx1.dtype != torch.int32 or idx2.dtype != torch.int32
            or a.size(1) == 0 or b.size(1) == 0 or tuple(idx1.shape) != tuple(a.shape[:2]) or tuple(idx2.shape) != tuple(b.shape[:2])):
        return None
    return MatchedPairLoss.apply(a, b, idx1, idx2, code)


def chamfer_min_keys(queries, refs, ref_offset):
    """One Chamfer direction against a local slice of the reference set -> packed int64 keys (B,Nq)."""
    _require_f32_contig(queries, "queries")
    _require_f32_contig(refs, "refs")
    _require_cuda(queries, "chamfer_min_keys")
    b, nq, _ = queries.shape
    nr = refs.size(1)
    with _on(queries.device):
        keys = torch.empty((b, nq), dtype=torch.int64, device=queries.device)
        rc = _native.lib().pdae_chamfer_min_keys_u64(queries.data_ptr(), refs.data_ptr(), b, nq, nr, int(ref_offset),
                                                     keys.data_ptr(), _stream())
    _native.check(rc, "pdae_chamfer_min_keys_u64")
    return keys


def chamfer_sharded_local(xyz1, xyz2_local, ref_offset, out_keys=None):
    """One rank's share of a reference-set-sharded forward in a single pass (every pair evaluated once):
    -> (keys1 (B,N) int64 for the MIN all-reduce, dist2_local (B,Ml) f32, idx2_local (B,Ml) int32).
    out_keys: an int64 (B,N) buffer to write the keys into (e.g. a view of a symmetric allocation)."""
    _require_f32_contig(xyz1, "xyz1")
    _require_f32_contig(xyz2_local, "xyz2_local")
    _require_cuda(xyz1, "chamfer_sharded_local")
    b, n, _ = xyz1.shape
    ml = xyz2_local.size(1)
    dev = xyz1.device
    with _on(dev):
        if out_keys is not None:
            if out_keys.dtype != torch.int64 or tuple(out_keys.shape) != (b, n) or not out_keys.is_contiguous() or out_keys.device != dev:
                raise RuntimeError("out_keys must be a contiguous int64 (B,N) tensor on xyz1's device")
            keys = out_keys
        else:
            keys = torch.empty((b, n), dtype=torch.int64, device=dev)
        d2 = torch.empty((b, ml), dtype=torch.float32, device=dev)
        i2 = torch.empty((b, ml), dtype=torch.int32, device=dev)
        nbytes = b * ml * 8
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        rc = _native.lib().pdae_chamfer_sharded_f32(xyz1.data_ptr(), xyz2_local.data_ptr(), b, n, ml, int(ref_offset),
                                                    keys.data_ptr(), d2.data_ptr(), i2.data_ptr(), ws.data_ptr(), nbytes,
                                                    _stream())
    _native.check(rc, "pdae_chamfer_sharded_f32")
    return keys, d2, i2


def chamfer_unpack_keys(keys):
    keys = keys.contiguous()
    with _on(keys.device):
        dist = torch.empty(keys.shape, dtype=torch.float32, device=keys.device)
        idx = torch.empty(keys.shape, dtype=torch.int32, device=keys.device)
        rc = _native.lib().pdae_chamfer_unpack_keys(keys.data_ptr(), keys.numel(), dist.data_ptr(), idx.data_ptr(),
                                                    _stream())
    _native.check(rc, "pdae_chamfer_unpack_keys")
    return dist, idx


# ---------------------------------------------------------------------------------------- DGCNN
def feat_knn(x, k):
    """models/dgcnn_util.py:7-12 `knn`: x (B,C,N) -> idx (B,N,k) int64."""
    _require_cuda(x, "knn")
    xc = x.detach()
    if xc.dtype != torch.float32 or not xc.is_contiguous():
        xc = xc.float().contiguous()
    b, c, n = xc.shape
    k = int(k)
    if not (1 <= k <= n):
        raise RuntimeError("selected index k out of range")  # torch.topk's message
    with _on(xc.device):
        idx = torch.empty((b, n, k), dtype=torch.int64, device=xc.device)
        L = _native.lib()
        nbytes = L.pdae_feat_knn_workspace_bytes(b, c, n, k)  # > 0: distance-matrix path (wide layers, k <= 32)
        if nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=xc.device)
            rc = L.pdae_feat_knn_ws_f32(xc.data_ptr(), b, c, n, k, idx.data_ptr(), ws.data_ptr(), nbytes, _stream())
        else:
            rc = L.pdae_feat_knn_f32(xc.data_ptr(), b, c, n, k, idx.data_ptr(), _stream())
    _native.check(rc, "pdae_feat_knn_f32")
    return idx


def _graph_feature_fwd(x, idx):
    b, c, n = x.shape
    k = idx.size(2)
    L = _native.lib()
    with _on(x.device):
        out = torch.empty((b, n, k, 2 * c), dtype=torch.float32, device=x.device)
        nbytes = L.pdae_graph_feature_workspace_bytes(b, c, n)
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=x.device)
        rc = L.pdae_graph_feature_f32(x.data_ptr(), idx.data_ptr(), b, c, n, k, out.data_ptr(), ws.data_ptr(), nbytes,
                                      _stream())
    _native.check(rc, "pdae_graph_feature_f32")
    return out


def _graph_feature_bwd(gout_phys, idx, c, n):
    b = gout_phys.size(0)
    k = idx.size(2)
    L = _native.lib()
    with _on(gout_phys.device):
        gx = torch.empty((b, c, n), dtype=torch.float32, device=gout_phys.device)
        det = _deterministic()
        nbytes = L.pdae_graph_feature_grad_det_workspace_bytes(b, c, n, k) if det else L.pdae_graph_feature_workspace_bytes(b, c, n)
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=gout_phys.device)
        grad = L.pdae_graph_feature_grad_det_f32 if det else L.pdae_graph_feature_grad_f32
        rc = grad(gout_phys.data_ptr(), idx.data_ptr(), b, c, n, k, gx.data_ptr(), ws.data_ptr(), nbytes, _stream())
    _native.check(rc, "pdae_graph_feature_grad_f32")
    return gx


class GraphFeatureFunction(torch.autograd.Function):
    """x (B,C,N) f32, idx (B,N,k) int64 per-cloud -> (B,2C,N,k) view of a (B,N,k,2C) tensor."""

    @staticmethod
    def forward(ctx, x, idx):
        xc = x.contiguous()
        ctx.save_for_backward(idx)
        ctx.cn = (xc.size(1), xc.size(2))
        return _graph_feature_fwd(xc, idx).permute(0, 3, 1, 2)

    @staticmethod
    def backward(ctx, grad):
        (idx,) = ctx.saved_tensors
        c, n = ctx.cn
        g = grad.permute(0, 2, 3, 1).contiguous().float()
        return _graph_feature_bwd(g, idx, c, n), None


# ---------------------------------------------------------------- EdgeConv, eval mode (SURVEY.md 8f row 4, stage 1)
def conv1x1(x, w, in_point_major=False, out_point_major=False, bias=None):
    """z[b,j,n] = sum_c w[j,c] x[b,c,n] (+ bias[j]) on the tensor cores (tcgen05 kind::tf32, 3xTF32 split: fp32 accuracy).
    x (B,C,N) -- or (B,N,C) with in_point_major --, w (J,C) f32 contiguous -> (B,J,N), or (B,N,J) with out_point_major."""
    _require_cuda(x, "conv1x1")
    _require_f32_contig(x, "x")
    _require_f32_contig(w, "w")
    _same_device(x.device, w=w)
    if in_point_major:
        b, n, c = x.shape
    else:
        b, c, n = x.shape
    j = w.size(0)
    if w.dim() != 2 or w.size(1) != c:
        raise RuntimeError("w must have shape (J, %d), got %s" % (c, tuple(w.shape)))
    L = _native.lib()
    with _on(x.device):
        z = torch.empty((b, n, j) if out_point_major else (b, j, n), dtype=torch.float32, device=x.device)
        nbytes = int(L.pdae_conv1x1_workspace_bytes(c, j))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
        if bias is not None:
            _require_f32_contig(bias, "bias")
            _same_device(x.device, bias=bias)
            if bias.numel() != j:
                raise RuntimeError("bias must have %d elements" % j)
        rc = L.pdae_conv1x1_tf32x3_f32(x.data_ptr(), w.data_ptr(), bias.data_ptr() if bias is not None else None, b, c, n, j,
                                       1 if in_point_major else 0,
                                       1 if out_point_major else 0, z.data_ptr(), ws.data_ptr(), nbytes, _stream())
    _native.check(rc, "pdae_conv1x1_tf32x3_f32")
    return z


class Conv1x1Function(torch.autograd.Function):
    """nn.Conv1d(C, J, 1) on point-major activations: x (N,C), weight (J,C), bias (J)|None -> (N,J); forward and the input
    gradient on the tensor cores, the (J x C) weight gradient as one plain library product."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x, weight = x.contiguous(), weight.contiguous()
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return conv1x1(x.unsqueeze(0), weight, True, True, bias.contiguous() if bias is not None else None).squeeze(0)

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        g = g.contiguous()
        dx = conv1x1(g.unsqueeze(0), weight.t().contiguous(), True, True).squeeze(0) if ctx.needs_input_grad[0] else None
        dw = torch.matmul(g.t(), x) if ctx.needs_input_grad[1] else None
        db = g.sum(dim=0) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return dx, dw, db


def pointwise_conv(x, conv):
    """x (N,C) point-major through an nn.Conv1d(C, J, kernel_size=1) -> (N,J)"""
    return Conv1x1Function.apply(x.float(), conv.weight.reshape(conv.out_channels, -1).float(),
                                 conv.bias.float() if conv.bias is not None else None)


def _edge_dims(z, idx, co):
    _require_cuda(z, "edge_conv")
    _require_f32_contig(z, "z")
    if idx.dtype != torch.int64 or not idx.is_contiguous() or idx.device != z.device:
        raise RuntimeError("idx must be a contiguous int64 tensor on z's device")
    b, n, ld = z.shape
    k = idx.size(2)
    if tuple(idx.shape[:2]) != (b, n) or ld < 2 * co or not (1 <= k <= 255):
        raise RuntimeError("edge_conv: z %s / idx %s / co=%d do not match" % (tuple(z.shape), tuple(idx.shape), co))
    return b, n, ld, k


def edge_stats(z, idx, co, want_s1=False):
    """Sum and sum of squares per output channel of y[i][j] = P[idx(i,j)] + Q[i] over all edges of the batch, from the
    point-major product z = [P | Q] (B,N,2*co): float64 (co, 2) (+ s1 (B,N,co) = sum_j P[idx(i,j)] for the backward)."""
    b, n, ld, k = _edge_dims(z, idx, co)
    L = _native.lib()
    with _on(z.device):
        partial = torch.empty((int(L.pdae_edge_partial_count(b, n)), co, 2), dtype=torch.float64, device=z.device)
        s1 = torch.empty((b, n, co), dtype=torch.float32, device=z.device) if want_s1 else None
        rc = L.pdae_edge_stats_f64(z.data_ptr(), ld, idx.data_ptr(), b, n, k, co, partial.data_ptr(),
                                   s1.data_ptr() if want_s1 else None, _stream())
    _native.check(rc, "pdae_edge_stats_f64")
    sums = partial.sum(dim=0)  # fixed order: deterministic
    return (sums, s1) if want_s1 else sums


def edge_forward(z, idx, co, scale, shift, slope=0.2, want_jstar=False):
    """out (B,co,N) = LeakyReLU(scale * (ext_j P[idx] + Q) + shift) (+ the selected neighbour slots (B,N,co) uint8)."""
    b, n, ld, k = _edge_dims(z, idx, co)
    _require_f32_contig(scale, "scale")
    _require_f32_contig(shift, "shift")
    with _on(z.device):
        out = torch.empty((b, co, n), dtype=torch.float32, device=z.device)
        jstar = torch.empty((b, n, co), dtype=torch.uint8, device=z.device) if want_jstar else None
        rc = _native.lib().pdae_edge_forward_f32(z.data_ptr(), ld, idx.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                                                 float(slope), b, n, k, co, out.data_ptr(),
                                                 jstar.data_ptr() if want_jstar else None, _stream())
    _native.check(rc, "pdae_edge_forward_f32")
    return out, jstar


def edge_backward(z, idx, co, jstar, g_pm, scale, shift, mean, invstd, gamma, slope, train, s1=None):
    """Backward of edge_forward (+ training-mode BatchNorm when train): g_pm (B,N,co) upstream gradient, point-major ->
    dz (B,N,ld) = [dP | dQ], dgamma (co), dbeta (co).  With s1 (sum_j P[idx], kept by the training forward) the dense
    terms of training-mode BatchNorm are gathered along the reversed graph (no float atomic per edge); without it the
    edge-parallel kernel of the first version runs."""
    b, n, ld, k = _edge_dims(z, idx, co)
    L = _native.lib()
    m = float(b) * n * k
    with _on(z.device):
        partial = torch.empty((int(L.pdae_edge_partial_count(b, n)), co, 2), dtype=torch.float64, device=z.device)
        dz = torch.zeros_like(z)
        if not train or s1 is not None:
            rc = L.pdae_edge_backward_select_f32(z.data_ptr(), ld, idx.data_ptr(), jstar.data_ptr(), g_pm.data_ptr(), scale.data_ptr(),
                                                 shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), float(slope),
                                                 1 if train else 0, b, n, k, co, partial.data_ptr(), dz.data_ptr(), _stream())
            _native.check(rc, "pdae_edge_backward_select_f32")
            sums = partial.sum(dim=0)
            dbeta, dgamma = sums[:, 0], sums[:, 1]
            if train:
                ca = (gamma.double() * dbeta / m).float().contiguous()
                cb = (gamma.double() * dgamma / m).float().contiguous()
                nints = int(L.pdae_edge_reverse_workspace_ints(b, n, k))
                ws = torch.empty(nints, dtype=torch.int32, device=z.device)
                rc = L.pdae_edge_backward_dense_f32(z.data_ptr(), ld, idx.data_ptr(), s1.data_ptr(), mean.data_ptr(), invstd.data_ptr(),
                                                    ca.data_ptr(), cb.data_ptr(), b, n, k, co, ws.data_ptr(), nints, dz.data_ptr(),
                                                    _stream())
                _native.check(rc, "pdae_edge_backward_dense_f32")
            return dz, dgamma.float(), dbeta.float()
        args = (z.data_ptr(), ld, idx.data_ptr(), jstar.data_ptr(), g_pm.data_ptr(), scale.data_ptr(), shift.data_ptr(),
                mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr())
        rc = L.pdae_edge_backward_f32(*args, None, None, float(slope), 1, b, n, k, co, partial.data_ptr(), None, _stream())
        _native.check(rc, "pdae_edge_backward_f32 (reduce)")
        sums = partial.sum(dim=0)
        dbeta, dgamma = sums[:, 0], sums[:, 1]
        ca = (gamma.double() * dbeta / m).float().contiguous()
        cb = (gamma.double() * dgamma / m).float().contiguous()
        rc = L.pdae_edge_backward_f32(*args, ca.data_ptr(), cb.data_ptr(), float(slope), 1, b, n, k, co, None, dz.data_ptr(), _stream())
    _native.check(rc, "pdae_edge_backward_f32")
    return dz, dgamma.float(), dbeta.float()


def _edge_partials(z, idx, co, want_s1):
    """raw per-CTA partial sums of the statistics kernel (summed inside pdae_edge_bn_prepare_f32)"""
    b, n, ld, k = _edge_dims(z, idx, co)
    L = _native.lib()
    partial = torch.empty((int(L.pdae_edge_partial_count(b, n)), co, 2), dtype=torch.float64, device=z.device)
    s1 = torch.empty((b, n, co), dtype=torch.float32, device=z.device) if want_s1 else None
    rc = L.pdae_edge_stats_f64(z.data_ptr(), ld, idx.data_ptr(), b, n, k, co, partial.data_ptr(),
                               s1.data_ptr() if want_s1 else None, _stream())
    _native.check(rc, "pdae_edge_stats_f64")
    return partial, s1


class EdgeConvFunction(torch.autograd.Function):
    """One EdgeConv layer of the DGCNN encoder (models/dgcnn_util.py:114-116 and the three after it):
    get_graph_feature(x, k, idx) -> Conv2d(2C, Co, 1, bias=False) -> BatchNorm2d -> LeakyReLU -> max over k, as
    tensor-core product + gather kernels; the (B,2C,N,k) and (B,Co,N,k) tensors never exist.  Training-mode BatchNorm
    takes its batch statistics from gather sums and updates the running buffers like nn.BatchNorm2d.  Host side: five
    launches forward, six backward, the per-channel arithmetic inside two of them (no torch micro-ops)."""

    @staticmethod
    def forward(ctx, x, idx, wz, gamma, beta, running_mean, running_var, training, momentum, eps, slope):
        co = wz.size(0) // 2
        b, c, n = x.shape
        k = idx.size(2)
        x = x.contiguous()
        L = _native.lib()
        need_grad = any(ctx.needs_input_grad)
        with _on(x.device):
            z = conv1x1(x, wz.contiguous(), out_point_major=True)  # (B,N,2co): [W1 x | (W2 - W1) x]
            partial = s1 = None
            if training:
                partial, s1 = _edge_partials(z, idx, co, need_grad)
            stats = torch.empty((4, co), dtype=torch.float32, device=x.device)  # mean | invstd | scale | shift
            gamma_c, beta_c = gamma.contiguous(), beta.contiguous()
            rc = L.pdae_edge_bn_prepare_f32(partial.data_ptr() if training else None, partial.size(0) if training else 0, co,
                                            float(b) * n * k, gamma_c.data_ptr(), beta_c.data_ptr(),
                                            running_mean.data_ptr() if running_mean is not None else None,
                                            running_var.data_ptr() if running_var is not None else None, float(momentum),
                                            float(eps), 1 if training else 0, stats[0].data_ptr(), stats[1].data_ptr(),
                                            stats[2].data_ptr(), stats[3].data_ptr(), _stream())
            _native.check(rc, "pdae_edge_bn_prepare_f32")
            out, jstar = edge_forward(z, idx, co, stats[2], stats[3], slope, want_jstar=need_grad)
        if need_grad:
            ctx.save_for_backward(x, idx, wz, z, jstar, stats, gamma_c, s1)
            ctx.meta = (co, float(slope), bool(training))
        return out

    @staticmethod
    def backward(ctx, g_out):
        x, idx, wz, z, jstar, stats, gamma, s1 = ctx.saved_tensors
        co, slope, training = ctx.meta
        b, n, ld, k = _edge_dims(z, idx, co)
        L = _native.lib()
        with _on(z.device):
            g_pm = g_out.transpose(1, 2).contiguous()
            mean, invstd, scale, shift = stats[0], stats[1], stats[2], stats[3]
            partial = torch.empty((int(L.pdae_edge_partial_count(b, n)), co, 2), dtype=torch.float64, device=z.device)
            dz = torch.zeros_like(z)
            rc = L.pdae_edge_backward_select_f32(z.data_ptr(), ld, idx.data_ptr(), jstar.data_ptr(), g_pm.data_ptr(), scale.data_ptr(),
                                                 shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), gamma.data_ptr(), slope,
                                                 1 if training else 0, b, n, k, co, partial.data_ptr(), dz.data_ptr(), _stream())
            _native.check(rc, "pdae_edge_backward_select_f32")
            grads = torch.empty((4, co), dtype=torch.float32, device=z.device)  # dgamma | dbeta | ca | cb
            rc = L.pdae_edge_bn_backward_f32(partial.data_ptr(), partial.size(0), co, float(b) * n * k, gamma.data_ptr(),
                                             grads[0].data_ptr(), grads[1].data_ptr(), grads[2].data_ptr(), grads[3].data_ptr(),
                                             _stream())
            _native.check(rc, "pdae_edge_bn_backward_f32")
            if training:
                nints = int(L.pdae_edge_reverse_workspace_ints(b, n, k))
                ws = torch.empty(nints, dtype=torch.int32, device=z.device)
                rc = L.pdae_edge_backward_dense_f32(z.data_ptr(), ld, idx.data_ptr(), s1.data_ptr(), mean.data_ptr(), invstd.data_ptr(),
                                                    grads[2].data_ptr(), grads[3].data_ptr(), b, n, k, co, ws.data_ptr(), nints,
                                                    dz.data_ptr(), _stream())
                _native.check(rc, "pdae_edge_backward_dense_f32")
            dx = dwz = None
            if ctx.needs_input_grad[0]:
                dx = conv1x1(dz, wz.t().contiguous(), in_point_major=True)  # (B,C,N) = Wz^T [dP ; dQ]
            if ctx.needs_input_grad[2]:
                c = x.size(1)
                # weight gradient: a (2co x B N) by (B N x C) product with a tiny output -- a plain library GEMM
                dwz = torch.matmul(dz.reshape(b * n, 2 * co).t(), x.transpose(1, 2).reshape(b * n, c))
        return dx, None, dwz, grads[0] if ctx.needs_input_grad[3] else None, grads[1] if ctx.needs_input_grad[4] else None, \
            None, None, None, None, None, None


def edge_conv(x, idx, weight, bn, slope=0.2):
    """x (B,C,N), idx (B,N,k) per-cloud int64, weight (Co,2C) (the layer's 1x1 convolution, bias-free), bn the layer's
    BatchNorm2d (its mode decides batch vs running statistics) -> (B,Co,N), differentiable w.r.t. x, weight, bn.weight,
    bn.bias."""
    c = x.size(1)
    w = weight.reshape(weight.size(0), -1).float()
    wz = torch.cat([w[:, :c], w[:, c:] - w[:, :c]], dim=0)  # differentiable: autograd maps d(wz) back to W1 / W2
    train_stats = bn.training or bn.running_mean is None
    momentum = 0.0 if bn.momentum is None else bn.momentum
    if bn.training and bn.track_running_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
        if bn.momentum is None:
            momentum = 1.0 / float(bn.num_batches_tracked)
    gamma = bn.weight if bn.weight is not None else torch.ones(w.size(0), device=x.device)
    beta = bn.bias if bn.bias is not None else torch.zeros(w.size(0), device=x.device)
    return EdgeConvFunction.apply(x.float(), idx.contiguous(), wz, gamma.float(), beta.float(),
                                  bn.running_mean if bn.track_running_stats else None,
                                  bn.running_var if bn.track_running_stats else None, train_stats, momentum, bn.eps, slope)


def edge_gather_extremum(p, q, idx, scale, shift, slope=0.2):
    """p, q (B,N,Co) f32 contiguous, idx (B,N,k) int64, scale / shift (Co) -> (B,Co,N):
    act(scale * (max|min_j p[idx] + q) + shift), max where scale >= 0, min where scale < 0 (pdae_edge_gather_extremum_f32)."""
    _require_cuda(p, "edge_conv")
    for t_, name in ((p, "p"), (q, "q"), (scale, "scale"), (shift, "shift")):
        _require_f32_contig(t_, name)
    if idx.dtype != torch.int64 or not idx.is_contiguous():
        raise RuntimeError("idx must be a contiguous int64 tensor")
    b, n, co = p.shape
    k = idx.size(2)
    if tuple(q.shape) != (b, n, co) or tuple(idx.shape[:2]) != (b, n) or scale.numel() != co or shift.numel() != co:
        raise RuntimeError("edge_gather_extremum: shapes do not match")
    with _on(p.device):
        out = torch.empty((b, co, n), dtype=torch.float32, device=p.device)
        rc = _native.lib().pdae_edge_gather_extremum_f32(p.data_ptr(), q.data_ptr(), idx.data_ptr(), scale.data_ptr(),
                                                         shift.data_ptr(), float(slope), b, n, k, co, out.data_ptr(), _stream())
    _native.check(rc, "pdae_edge_gather_extremum_f32")
    return out


def edge_conv_max(x, idx, weight, scale, shift, slope=0.2):
    """One eval-mode EdgeConv layer (models/dgcnn_util.py:114-126) without the k-replicated tensors: x (B,C,N), idx (B,N,k)
    per-cloud int64, weight (Co,2C) of the 1x1 convolution, BatchNorm folded to scale / shift (Co) -> (B,Co,N).
    The tensor-core product [P | Q] = x^T [W1 ; W2 - W1]^T (conv1x1) + the gather kernel.  No gradient: the
    differentiable, training-capable form is `edge_conv`."""
    c = x.size(1)
    co = weight.size(0)
    with torch.no_grad():
        w = weight.reshape(co, -1).float()
        wz = torch.cat([w[:, :c], w[:, c:] - w[:, :c]], dim=0).contiguous()
        z = conv1x1(x.detach().float().contiguous(), wz, out_point_major=True)
        return edge_forward(z, idx.contiguous(), co, scale.float().contiguous(), shift.float().contiguous(), slope)[0]


# ---------------------------------------------------------------------------- ball query / group
def ball_query(new_xyz, xyz, radius, nsample):
    """pointnet2._ext.ball_query(new_xyz (B,M,3), xyz (B,N,3), radius, nsample) -> (B,M,nsample) int32."""
    _require_f32_contig(new_xyz, "new_xyz")
    _require_f32_contig(xyz, "xyz")
    _require_cuda(new_xyz, "ball_query")
    _require_cuda(xyz, "ball_query")
    b, m, _ = new_xyz.shape
    n = xyz.size(1)
    with _on(xyz.device):
        idx = torch.empty((b, m, int(nsample)), dtype=torch.int32, device=xyz.device)
        rc = _native.lib().pdae_ball_query_f32(new_xyz.data_ptr(), xyz.data_ptr(), b, n, m, float(radius),
                                               int(nsample), idx.data_ptr(), _stream())
    _native.check(rc, "pdae_ball_query_f32")
    return idx


def group_points(points, idx):
    """pointnet2._ext.group_points(points (B,C,N), idx (B,P,S) int32) -> (B,C,P,S)."""
    _require_f32_contig(points, "points")
    _require_i32_contig(idx, "idx")
    _require_cuda(points, "group_points")
    _require_cuda(idx, "group_points")
    b, c, n = points.shape
    _, p, s = idx.shape
    with _on(points.device):
        out = torch.empty((b, c, p, s), dtype=torch.float32, device=points.device)
        rc = _native.lib().pdae_group_points_f32(points.data_ptr(), idx.data_ptr(), b, c, n, p, s, out.data_ptr(),
                                                 _stream())
    _native.check(rc, "pdae_group_points_f32")
    return out


def group_points_grad(grad_out, idx, n):
    _require_f32_contig(grad_out, "grad_out")
    _require_i32_contig(idx, "idx")
    _require_cuda(grad_out, "group_points_grad")
    b, c, p, s = grad_out.shape
    with _on(grad_out.device):
        out = torch.empty((b, c, int(n)), dtype=torch.float32, device=grad_out.device)
        L = _native.lib()
        if _deterministic():
            nbytes = L.pdae_group_points_grad_det_workspace_bytes(b, int(n), p, s)
            ws = _workspace(nbytes, grad_out.device)
            rc = L.pdae_group_points_grad_det_f32(grad_out.data_ptr(), idx.data_ptr(), b, c, int(n), p, s, out.data_ptr(),
                                                  ws.data_ptr(), nbytes, _stream())
        else:
            rc = L.pdae_group_points_grad_f32(grad_out.data_ptr(), idx.data_ptr(), b, c, int(n), p, s, out.data_ptr(),
                                              _stream())
    _native.check(rc, "pdae_group_points_grad_f32")
    return out


# ------------------------------------------------------------------- three_nn / three_interpolate
def three_nn(unknown, known):
    """pointnet2._ext.three_nn(unknown (B,n,3), known (B,m,3)) -> [dist2 (B,n,3) squared, idx (B,n,3) int32]
    (interpolate.cpp:17-46)."""
    _require_f32_contig(unknown, "unknowns")
    _require_f32_contig(known, "knows")
    _require_cuda(unknown, "three_nn")
    _require_cuda(known, "three_nn")
    b, n, _ = unknown.shape
    m = known.size(1)
    with _on(unknown.device):
        dist2 = torch.empty((b, n, 3), dtype=torch.float32, device=unknown.device)
        idx = torch.empty((b, n, 3), dtype=torch.int32, device=unknown.device)
        rc = _native.lib().pdae_three_nn_f32(unknown.data_ptr(), known.data_ptr(), b, n, m, dist2.data_ptr(),
                                             idx.data_ptr(), _stream())
    _native.check(rc, "pdae_three_nn_f32")
    return [dist2, idx]


def three_interpolate(points, idx, weight):
    """pointnet2._ext.three_interpolate(points (B,c,m), idx (B,n,3) int32, weight (B,n,3)) -> (B,c,n)
    (interpolate.cpp:48-77)."""
    _require_f32_contig(points, "points")
    _require_i32_contig(idx, "idx")
    _require_f32_contig(weight, "weight")
    for t in (points, idx, weight):
        _require_cuda(t, "three_interpolate")
    b, c, m = points.shape
    n = idx.size(1)
    with _on(points.device):
        out = torch.empty((b, c, n), dtype=torch.float32, device=points.device)
        rc = _native.lib().pdae_three_interpolate_f32(points.data_ptr(), idx.data_ptr(), weight.data_ptr(), b, c, m, n,
                                                      out.data_ptr(), _stream())
    _native.check(rc, "pdae_three_interpolate_f32")
    return out


def three_interpolate_grad(grad_out, idx, weight, m):
    """pointnet2._ext.three_interpolate_grad(grad_out (B,c,n), idx, weight, m) -> (B,c,m) (interpolate.cpp:78-106)."""
    _require_f32_contig(grad_out, "grad_out")
    _require_i32_contig(idx, "idx")
    _require_f32_contig(weight, "weight")
    for t in (grad_out, idx, weight):
        _require_cuda(t, "three_interpolate_grad")
    b, c, n = grad_out.shape
    with _on(grad_out.device):
        out = torch.empty((b, c, int(m)), dtype=torch.float32, device=grad_out.device)
        L = _native.lib()
        if _deterministic():
            nbytes = L.pdae_three_interpolate_grad_det_workspace_bytes(b, n, int(m))
            ws = _workspace(nbytes, grad_out.device)
            rc = L.pdae_three_interpolate_grad_det_f32(grad_out.data_ptr(), idx.data_ptr(), weight.data_ptr(), b, c, n, int(m),
                                                       out.data_ptr(), ws.data_ptr(), nbytes, _stream())
        else:
            rc = L.pdae_three_interpolate_grad_f32(grad_out.data_ptr(), idx.data_ptr(), weight.data_ptr(), b, c, n, int(m),
                                                   out.data_ptr(), _stream())
    _native.check(rc, "pdae_three_interpolate_grad_f32")
    return out


# ------------------------------------------------------------------- Earth Mover's Distance (approxmatch)
EMD_LEVELS = 10


def _emd_clouds(xyz1, xyz2, name):
    for t, nm in ((xyz1, "xyz1"), (xyz2, "xyz2")):
        _require_cuda(t, name)
        _require_f32_contig(t, nm)
        if t.dim() != 3 or t.size(2) != 3:
            raise RuntimeError("%s must have shape (B, N, 3)" % nm)
    _same_device(xyz1.device, xyz2=xyz2)
    if xyz1.size(0) != xyz2.size(0):
        raise RuntimeError("xyz1 and xyz2 disagree on the batch size")
    return xyz1.shape[0], xyz1.shape[1], xyz2.shape[1]


def _emd_inputs(xyz1, xyz2, name, match, ratio_l, ratio_r):
    """checks the clouds and the match or ratios; -> (b, n, m, pointers of match / ratio_l / ratio_r or None)"""
    b, n, m = _emd_clouds(xyz1, xyz2, name)
    if match is not None:
        _require_f32_contig(match, "match")
        _same_device(xyz1.device, match=match)
        if tuple(match.shape) != (b, m, n):
            raise RuntimeError("match must have shape (B, m, n) = (%d, %d, %d)" % (b, m, n))
        return b, n, m, (match.data_ptr(), None, None)
    if ratio_l is None or ratio_r is None:
        raise RuntimeError("%s needs either match or both ratios" % name)
    for t, nm, cnt in ((ratio_l, "ratio_l", n), (ratio_r, "ratio_r", m)):
        _require_f32_contig(t, nm)
        _same_device(xyz1.device, **{nm: t})
        if tuple(t.shape) != (b, EMD_LEVELS, cnt):
            raise RuntimeError("%s must have shape (B, %d, %d)" % (nm, EMD_LEVELS, cnt))
    return b, n, m, (None, ratio_l.data_ptr(), ratio_r.data_ptr())


def emd_match(xyz1, xyz2, materialize=False):
    """approxmatch of xyz1 (B,n,3) and xyz2 (B,m,3): -> (ratio_l (B,10,n), ratio_r (B,10,m), match (B,m,n) or None).
    The per-level ratios determine the match; it is written only with materialize=True."""
    b, n, m = _emd_clouds(xyz1, xyz2, "emd_match")
    dev = xyz1.device
    L = _native.lib()
    with _on(dev):
        ratio_l = torch.empty((b, EMD_LEVELS, n), dtype=torch.float32, device=dev)
        ratio_r = torch.empty((b, EMD_LEVELS, m), dtype=torch.float32, device=dev)
        match = torch.empty((b, m, n), dtype=torch.float32, device=dev) if materialize else None
        nbytes = L.pdae_emd_workspace_bytes(b, n, m)
        ws = _workspace(nbytes, dev)
        rc = L.pdae_emd_match_f32(xyz1.data_ptr(), xyz2.data_ptr(), b, n, m, ratio_l.data_ptr(), ratio_r.data_ptr(),
                                  match.data_ptr() if materialize else None, ws.data_ptr(), nbytes, _stream())
    _native.check(rc, "pdae_emd_match_f32")
    return ratio_l, ratio_r, match


def emd_cost(xyz1, xyz2, match=None, ratio_l=None, ratio_r=None):
    """matchcost: (B,) sum over pairs of |x1_k - x2_l| * match[l][k], the match given or rebuilt from the ratios."""
    b, n, m, (pm, pl, pr) = _emd_inputs(xyz1, xyz2, "emd_cost", match, ratio_l, ratio_r)
    dev = xyz1.device
    L = _native.lib()
    with _on(dev):
        cost = torch.empty((b,), dtype=torch.float32, device=dev)
        nbytes = L.pdae_emd_workspace_bytes(b, n, m)
        ws = _workspace(nbytes, dev)
        rc = L.pdae_emd_cost_f32(xyz1.data_ptr(), xyz2.data_ptr(), b, n, m, pm, pl, pr, cost.data_ptr(), ws.data_ptr(),
                                 nbytes, _stream())
    _native.check(rc, "pdae_emd_cost_f32")
    return cost


def emd_cost_grad(grad_cost, xyz1, xyz2, match=None, ratio_l=None, ratio_r=None):
    """matchcost gradient with the match held constant: grad_cost (B,) -> (grad1 (B,n,3), grad2 (B,m,3))."""
    b, n, m, (pm, pl, pr) = _emd_inputs(xyz1, xyz2, "emd_cost_grad", match, ratio_l, ratio_r)
    _require_cuda(grad_cost, "emd_cost_grad")
    _require_f32_contig(grad_cost, "grad_cost")
    _same_device(xyz1.device, grad_cost=grad_cost)
    if grad_cost.numel() != b:
        raise RuntimeError("grad_cost must hold one value per cloud")
    dev = xyz1.device
    with _on(dev):
        grad1 = torch.empty((b, n, 3), dtype=torch.float32, device=dev)
        grad2 = torch.empty((b, m, 3), dtype=torch.float32, device=dev)
        rc = _native.lib().pdae_emd_cost_grad_f32(grad_cost.data_ptr(), xyz1.data_ptr(), xyz2.data_ptr(), b, n, m, pm, pl,
                                                  pr, grad1.data_ptr(), grad2.data_ptr(), _stream())
    _native.check(rc, "pdae_emd_cost_grad_f32")
    return grad1, grad2


# ------------------------------------------------- variable-size clouds in one batch (the reference's pointops)
def _segment_inputs(xyz, offset, new_offset, name):
    _require_cuda(xyz, name)
    _require_f32_contig(xyz, "xyz")
    if xyz.dim() != 2 or xyz.size(1) != 3:
        raise RuntimeError("xyz must have shape (N, 3)")
    for t, nm in ((offset, "offset"), (new_offset, "new_offset")):
        _require_i32_contig(t, nm)
        if t.dim() != 1:
            raise RuntimeError("%s must have shape (b,)" % nm)
    _same_device(xyz.device, offset=offset, new_offset=new_offset)
    if offset.numel() != new_offset.numel():
        raise RuntimeError("offset and new_offset disagree on the number of segments")
    return offset.numel()


def segment_fps_into(xyz, offset, new_offset, n, idx, tmp=None):
    """The compiled pointops FPS: writes the global sample indices of every segment into idx (M,) int32 and, when tmp
    (N,) fp32 is given, starts from and leaves the running minima there.  n (the largest segment size) sets the tie
    rule; segments larger than n are still exact.  No host synchronisation."""
    b = _segment_inputs(xyz, offset, new_offset, "furthestsampling")
    _require_i32_contig(idx, "idx")
    _same_device(xyz.device, idx=idx, tmp=tmp)
    if tmp is not None:
        _require_f32_contig(tmp, "tmp")
        if tmp.numel() < xyz.size(0):
            raise RuntimeError("tmp must hold one value per point")
    n_total = xyz.size(0)
    L = _native.lib()
    with _on(xyz.device):
        nbytes = L.pdae_seg_fps_workspace_bytes(n_total) if tmp is None else 0
        ws = _workspace(nbytes, xyz.device) if nbytes else None
        rc = L.pdae_seg_fps_f32(xyz.data_ptr(), n_total, offset.data_ptr(), new_offset.data_ptr(), b, int(n), idx.numel(),
                                tmp.data_ptr() if tmp is not None else None, idx.data_ptr(),
                                ws.data_ptr() if ws is not None else None, nbytes, _stream())
    _native.check(rc, "pdae_seg_fps_f32")
    return idx


def segment_fps(xyz, offset, new_offset, n=None, m=None):
    """Furthest point sampling of every segment of a packed batch: xyz (N,3) f32, offset / new_offset (b,) int32
    cumulative ends of the points / samples -> idx (m,) int32 of global indices, m = new_offset[-1].

    n is the largest segment size (it sets the reference's tie rule) and m the number of samples.  Each one left as None
    is computed from the offsets on the host: this is the one host read of the call (one copy for both).  Pass both to
    keep the call free of synchronisation, e.g. inside a CUDA graph."""
    b = _segment_inputs(xyz, offset, new_offset, "segment_fps")
    if b == 0:
        return torch.empty((0 if m is None else int(m),), dtype=torch.int32, device=xyz.device)
    if n is None or m is None:
        with _on(xyz.device):
            sizes = torch.diff(offset, prepend=offset.new_zeros(1))
            n_read, m_read = torch.stack((sizes.max(), new_offset[-1])).tolist()
        n = n_read if n is None else n
        m = m_read if m is None else m
    with _on(xyz.device):
        idx = torch.empty((max(int(m), 0),), dtype=torch.int32, device=xyz.device)
    return segment_fps_into(xyz, offset, new_offset, max(int(n), 0), idx)


def segment_knn_into(nsample, xyz, new_xyz, offset, new_offset, idx, dist2):
    """The compiled pointops kNN query: writes idx (m, nsample) int32 and dist2 (m, nsample) fp32 (squared)."""
    b = _segment_inputs(xyz, offset, new_offset, "knnquery")
    _require_cuda(new_xyz, "knnquery")
    _require_f32_contig(new_xyz, "new_xyz")
    if new_xyz.dim() != 2 or new_xyz.size(1) != 3:
        raise RuntimeError("new_xyz must have shape (M, 3)")
    nsample = int(nsample)
    if not 1 <= nsample <= 100:
        raise RuntimeError("nsample=%d must satisfy 1 <= nsample <= 100" % nsample)
    m = new_xyz.size(0)
    _require_i32_contig(idx, "idx")
    _require_f32_contig(dist2, "dist2")
    _same_device(xyz.device, new_xyz=new_xyz, idx=idx, dist2=dist2)
    if idx.numel() != m * nsample or dist2.numel() != m * nsample:
        raise RuntimeError("idx and dist2 must hold (M, nsample) = (%d, %d) elements" % (m, nsample))
    L = _native.lib()
    with _on(xyz.device):
        nbytes = L.pdae_seg_knn_workspace_bytes(b, m)
        ws = _workspace(nbytes, xyz.device)
        rc = L.pdae_seg_knn_f32(xyz.data_ptr(), xyz.size(0), new_xyz.data_ptr(), m, offset.data_ptr(), new_offset.data_ptr(),
                                b, nsample, idx.data_ptr(), dist2.data_ptr(), ws.data_ptr(), nbytes, _stream())
    _native.check(rc, "pdae_seg_knn_f32")
    return idx, dist2


def segment_knn(nsample, xyz, new_xyz, offset, new_offset):
    """kNN of every query among the points of its own segment: xyz (N,3), new_xyz (M,3) f32, offset / new_offset (b,)
    int32 cumulative ends -> (idx (M,nsample) int32 global indices, dist2 (M,nsample) f32 squared distances), ascending
    by (distance, index).  Slots no point fills hold (start of the segment, 1e10); rows past new_offset[-1] hold
    (-1, 1e10).  1 <= nsample <= 100.  No host synchronisation."""
    m = new_xyz.size(0)
    with _on(xyz.device):
        idx = torch.empty((m, int(nsample)), dtype=torch.int32, device=xyz.device)
        dist2 = torch.empty((m, int(nsample)), dtype=torch.float32, device=xyz.device)
    return segment_knn_into(nsample, xyz, new_xyz, offset, new_offset, idx, dist2)
