"""ctypes binding of libpointdae_b200.so (the C ABI declared in include/pointdae_b200.h).

There is no CPU fallback and no alternative backend: if the library is missing this module
raises at first use, loudly.  ctypes releases the GIL for the duration of every call, so the
reference's nn.DataParallel threading model (one Python thread per GPU, tools/runner_pretrain.py:86-88)
does not serialise on launches.
"""
import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpointdae_b200.so")
BUILD_SH = os.path.join(_HERE, "csrc", "build.sh")

_vp, _i, _f, _sz, _ll = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t, ctypes.c_longlong

# name -> (restype, argtypes); must list every symbol include/pointdae_b200.h declares.
SIGNATURES = {
    "pdae_abi_version": (_i, []),
    "pdae_strerror": (ctypes.c_char_p, [_i]),
    "pdae_fps_block_size": (_i, [_i]),
    "pdae_fps_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_fps_f32": (_i, [_vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_fps_gather_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_gather_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pdae_gather_grad_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pdae_knn_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_chamfer_exchange_keys_peer": (_i, [_vp, _vp, _vp, _i, _ll, _ll, _vp]),
    "pdae_chamfer_exchange_keys_multimem": (_i, [_vp, _vp, _vp, _ll, _ll, _vp]),
    "pdae_knn_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "pdae_knn_ws_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_group_ws_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_knn_keys_u64": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _ll, _vp, _vp]),
    "pdae_knn_merge_keys_u64": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_group_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_fps_group_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pdae_fps_group_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_fps_group_ex_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, ctypes.c_uint, _vp]),
    "pdae_tune_patchify": (_i, [_i, _i, _i]),
    "pdae_step_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pdae_step_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_patchify_trace": (_i, [_vp]),
    "pdae_fps_group_affine_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_group_gather_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_feat_knn_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "pdae_feat_knn_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pdae_feat_knn_ws_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_graph_feature_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_graph_feature_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_graph_feature_grad_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_chamfer_fwd_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_chamfer_fwd_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_chamfer_fwd_phase_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _i, _vp]),
    "pdae_chamfer_bwd_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_conv1x1_workspace_bytes": (_sz, [_i, _i]),
    "pdae_conv1x1_tf32x3_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_edge_partial_count": (_sz, [_i, _i]),
    "pdae_edge_stats_f64": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_edge_bn_prepare_f32": (_i, [_vp, _i, _i, ctypes.c_double, _vp, _vp, _vp, _vp, _f, _f, _i, _vp, _vp, _vp, _vp, _vp]),
    "pdae_edge_stats_shifted_f64": (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_edge_bn_prepare_shifted_f32": (_i, [_vp, _i, _i, ctypes.c_double, _vp, _i, _vp, _vp, _vp, _vp, _f, _f, _i, _vp, _vp, _vp,
                                              _vp, _vp]),
    "pdae_edge_bn_backward_f32": (_i, [_vp, _i, _i, ctypes.c_double, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pdae_edge_reverse_workspace_ints": (_sz, [_i, _i, _i]),
    "pdae_edge_backward_select_f32": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_edge_backward_dense_f32": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp, _vp]),
    "pdae_edge_forward_f32": (_i, [_vp, _i, _vp, _vp, _vp, _f, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_edge_backward_f32": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_pair_loss_partial_count": (_sz, [_i, _i, _i]),
    "pdae_pair_loss_fwd_f64": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "pdae_pair_loss_bwd_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_tune_chamfer_split": (_i, [_i]),
    "pdae_tune_chamfer_tc": (_i, [_i, _f]),
    "pdae_chamfer_tc_probe": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pdae_tune_knn": (_i, [_i, _i, _i, _i]),
    "pdae_chamfer_tc_shares": (_i, [_i, _i, _i, _i, _vp, _vp]),
    "pdae_chamfer_loss_workspace_bytes": (_sz, []),
    "pdae_chamfer_loss_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_chamfer_loss_bwd_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_chamfer_min_keys_u64": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pdae_chamfer_unpack_keys": (_i, [_vp, _ll, _vp, _vp, _vp]),
    "pdae_chamfer_sharded_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_ball_query_f32": (_i, [_vp, _vp, _i, _i, _i, _f, _i, _vp, _vp]),
    "pdae_group_points_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "pdae_group_points_grad_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "pdae_three_nn_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_three_interpolate_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pdae_three_interpolate_grad_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "pdae_affine_points_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pdae_group_affine_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "pdae_edge_gather_extremum_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _vp, _vp]),
    "pdae_chamfer_bwd_det_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_chamfer_bwd_det_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_chamfer_loss_bwd_det_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_pair_loss_bwd_det_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_pair_loss_bwd_det_f32": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_gather_grad_det_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_gather_grad_det_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_group_points_grad_det_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pdae_group_points_grad_det_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_three_interpolate_grad_det_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_three_interpolate_grad_det_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_graph_feature_grad_det_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "pdae_graph_feature_grad_det_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "pdae_reverse_index_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_reverse_index_i32": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_reverse_index_i64": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_step_ex_workspace_bytes": (_sz, [_i, _i, _i, _i, ctypes.c_uint]),
    "pdae_step_ex_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz,
                              ctypes.c_uint, _vp]),
    "pdae_emd_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_emd_match_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_emd_cost_f32": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_emd_cost_grad_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pdae_seg_fps_workspace_bytes": (_sz, [_i]),
    "pdae_seg_fps_f32": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_knn_workspace_bytes": (_sz, [_i, _i]),
    "pdae_seg_knn_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_chamfer_fwd_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_seg_chamfer_fwd_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_chamfer_bwd_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pdae_seg_chamfer_bwd_det_workspace_bytes": (_sz, [_i, _i]),
    "pdae_seg_chamfer_bwd_det_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_chamfer_loss_workspace_bytes": (_sz, [_i]),
    "pdae_seg_chamfer_loss_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_chamfer_loss_bwd_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _vp]),
    "pdae_seg_chamfer_loss_bwd_det_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _sz,
                                               _vp]),
    "pdae_seg_emd_workspace_bytes": (_sz, [_i, _i, _i]),
    "pdae_seg_emd_match_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_emd_cost_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pdae_seg_emd_cost_grad_f32": (_i, [_vp, _vp, _i, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
}

_lib = None
_lock = threading.Lock()


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into lib/libpointdae_b200.so (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["sh", BUILD_SH], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout)
        print(out.stderr)
    if out.returncode != 0:
        raise RuntimeError("building libpointdae_b200.so failed:\n" + out.stderr[-4000:])
    return LIB_PATH


def lib():
    """The loaded library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "libpointdae_b200.so not found at %s -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(or sh point-dae_b200/csrc/build.sh).  There is no CPU fallback." % LIB_PATH)
                handle = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)  # AttributeError if the ABI lost a symbol
                    fn.restype = res
                    fn.argtypes = args
                if handle.pdae_abi_version() != 1:
                    raise RuntimeError("libpointdae_b200.so ABI version mismatch")
                _lib = handle
    return _lib


def check(code, what):
    if code != 0:
        msg = lib().pdae_strerror(code)
        raise RuntimeError("%s failed: %s (code %d)" % (what, msg.decode() if msg else "?", code))
