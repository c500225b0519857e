"""The C-ABI shared library loads and exports every symbol include/pointdae_b200.h declares
(no compute calls: this runs without a GPU)."""
import ctypes
import os
import re

import pytest

from pointdae_b200 import _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "pointdae_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pdae_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_hot_path():
    syms = declared_symbols()
    for need in ("pdae_fps_f32", "pdae_gather_f32", "pdae_gather_grad_f32", "pdae_knn_f32", "pdae_group_f32",
                 "pdae_feat_knn_f32", "pdae_graph_feature_f32", "pdae_graph_feature_grad_f32", "pdae_chamfer_fwd_f32",
                 "pdae_chamfer_bwd_f32", "pdae_chamfer_min_keys_u64"):
        assert need in syms


def test_library_exports_every_declared_symbol():
    if not os.path.exists(_native.LIB_PATH):
        _native.build()
    handle = ctypes.CDLL(_native.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(handle, name), "libpointdae_b200.so does not export %s" % name


def test_python_binding_covers_the_header():
    assert sorted(_native.SIGNATURES) == declared_symbols()


def test_host_only_entry_points():
    L = _native.lib()
    assert L.pdae_abi_version() == 1
    assert L.pdae_strerror(0) == b"success"
    assert b"invalid" in L.pdae_strerror(-1)
    assert L.pdae_fps_workspace_bytes(4, 2048, 64) == 0
    assert L.pdae_fps_workspace_bytes(2, 100000, 64) == 0  # cluster kernel: state stays on chip
    assert L.pdae_fps_workspace_bytes(2, 300000, 64) == 2 * 300000 * 4  # beyond a 16-CTA cluster: global running minima
    assert L.pdae_graph_feature_workspace_bytes(2, 64, 1024) == 2 * 64 * 1024 * 4


def test_argument_validation_needs_no_gpu():
    L = _native.lib()
    # negative sizes / null pointers are rejected before any CUDA call
    assert L.pdae_chamfer_fwd_f32(None, None, -1, 4, 4, None, None, None, None, None, 0, None) == -1
    assert L.pdae_chamfer_fwd_f32(None, None, 2, 4, 4, None, None, None, None, None, 0, None) == -1
    assert L.pdae_chamfer_fwd_workspace_bytes(2, 2048, 1024) == 2 * (2048 + 1024) * 8  # column keys + row keys
    assert L.pdae_knn_f32(None, None, 1, 8, 4, 3, 0, 0, None, None, None) == -1
    assert L.pdae_fps_f32(None, 0, 16, 4, None, None, 0, None) == 0  # empty batch is a no-op
    # affine corruptions: chain length 0..8, null pointers, empty batch
    assert L.pdae_affine_points_f32(None, None, None, 2, 4, 4, 9, None, None, None) == -1
    assert L.pdae_affine_points_f32(None, None, None, 2, 4, 4, 1, None, None, None) == -1
    assert L.pdae_affine_points_f32(None, None, None, 0, 4, 4, 1, None, None, None) == 0
    assert L.pdae_group_affine_f32(None, None, None, 2, 64, 4, 8, 1, None, None, None, None, None) == -1
    assert L.pdae_group_affine_f32(None, None, None, 0, 64, 4, 8, 1, None, None, None, None, None) == 0
    # the single-launch patchifier and the native step: null pointers, unknown launch flags, empty batch, workspace sizes
    assert L.pdae_fps_group_f32(None, 2, 1024, 64, 32, None, None, None, None, None, 0, None) == -1
    assert L.pdae_fps_group_ex_f32(None, 0, 1024, 64, 32, None, None, None, None, None, 0, 2, None) == -1  # flag 2 is not defined
    assert L.pdae_fps_group_ex_f32(None, 0, 1024, 64, 32, None, None, None, None, None, 0, 1, None) == 0
    assert L.pdae_fps_group_affine_f32(None, None, 2, 1024, 64, 32, 9, *([None] * 6), None, 0, None) == -1  # chain too long
    assert L.pdae_fps_group_workspace_bytes(128, 2048, 64, 32) == 0      # one launch, state in shared memory
    assert L.pdae_fps_group_workspace_bytes(1, 100000, 2048, 64) > 0     # two launches, chunked kNN merge
    assert L.pdae_step_f32(None, None, 0, 2048, 64, 32, *([None] * 11), None, 0, None) == 0
    assert L.pdae_step_f32(None, None, 2, 2048, 64, 32, *([None] * 11), None, 0, None) == -1
    assert L.pdae_step_workspace_bytes(128, 2048, 64, 32) % 256 == 0
    # kNN tuning hook: form -1 (automatic) or 0..3; anything else is rejected
    assert L.pdae_tune_knn(4, -1, -1, -1) == -1
    assert L.pdae_tune_knn(-2, -1, -1, -1) == -1


def test_source_is_sm100a_only():
    sh = open(os.path.join(ROOT, "point-dae_b200", "csrc", "build.sh")).read()
    assert "arch=compute_100a,code=sm_100a" in sh and "-lineinfo" in sh
