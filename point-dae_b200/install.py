"""`install()` makes the reference's imports resolve to this package, so Point-DAE's models/ and
main.py run unchanged:

    import pointdae_b200; pointdae_b200.install()
    # now: from pointnet2_ops import pointnet2_utils (and pointnet2_ops.pointnet2_modules) ; from knn_cuda import KNN ; import chamfer ;
    #      import pointnet2._ext ; import emd_cuda  -> all served by the sm_100a kernels

Only the *compiled / third-party* modules are replaced (the reference's own Python, e.g.
extensions/chamfer_dist/__init__.py, keeps running on top).  `patch_models()` additionally rebinds
the pure-torch hot functions that live inside the reference's packages (dgcnn knn / get_graph_feature,
misc.fps, Group) once those packages are importable.
"""
import importlib
import sys
import types


def install(loss_modules=False):
    """loss_modules=True additionally serves `extensions.chamfer_dist` (the reference's Python loss classes,
    which import `ipdb` at module level, extensions/chamfer_dist/__init__.py:12) from this package's mirror."""
    from . import chamfer, emd_cuda, knn_cuda, pointnet2_ext, pointnet2_modules, pointnet2_utils

    pkg = types.ModuleType("pointnet2_ops")
    pkg.__path__ = []  # mark as package
    pkg.pointnet2_utils = pointnet2_utils
    pkg.pointnet2_modules = pointnet2_modules  # models/pointnetv2_util.py:317, pulled in by `import models`
    pkg.__version__ = "3.0.0"
    sys.modules["pointnet2_ops"] = pkg
    sys.modules["pointnet2_ops.pointnet2_utils"] = pointnet2_utils
    sys.modules["pointnet2_ops.pointnet2_modules"] = pointnet2_modules

    sys.modules["knn_cuda"] = knn_cuda
    sys.modules["chamfer"] = chamfer
    sys.modules["emd_cuda"] = emd_cuda  # extensions/emd's compiled module

    # `import pointnet2._ext as _ext` (extensions/pointnet2/pointnet2_utils.py:23-24)
    p2 = sys.modules.get("pointnet2")
    if p2 is None:
        p2 = types.ModuleType("pointnet2")
        p2.__path__ = []
        sys.modules["pointnet2"] = p2
    p2._ext = pointnet2_ext
    sys.modules["pointnet2._ext"] = pointnet2_ext

    if loss_modules:
        from . import chamfer_dist
        ext = sys.modules.get("extensions")
        if ext is None:
            try:
                ext = importlib.import_module("extensions")
            except Exception:
                ext = types.ModuleType("extensions")
                ext.__path__ = []
                sys.modules["extensions"] = ext
        ext.chamfer_dist = chamfer_dist
        sys.modules["extensions.chamfer_dist"] = chamfer_dist
    return True


def patch_models(names=("models.dgcnn_util", "models.PointCAE_DGCNN", "segmentation.models.dgcnn_util"), edgeconv=True):
    """Rebind the pure-torch hot functions that live inside the reference's own packages: knn / get_graph_feature,
    misc.fps, the corruptions executed inside forward, and every flavour of the `Group` patchifier.  Names that other
    reference modules imported from the defining module (`from .Point_M2AE_modules import *`,
    `from datasets.corrupt_util_tensor import corrupt_data`) are rebound there too.  `edgeconv=True` (default) also routes
    `dgcnn_encoder.forward` through the fused tensor-core EdgeConv layers (training and eval, differentiable; GPU parity in
    tests/test_gpu_edgeconv_tc.py); `edgeconv=False` keeps the reference's layer sequence on this repo's knn / get_graph_feature.  Returns what was rebound."""
    from . import corrupt_util_tensor, dgcnn_util, group

    patched, replaced = [], {}

    def rebind(mod, attr, new, where):
        old = getattr(mod, attr, None)
        if old is None or old is new:
            return
        if callable(old):
            replaced[id(old)] = (old, new)
        setattr(mod, attr, new)
        patched.append(where + "." + attr)

    for name in names:
        try:
            mod = importlib.import_module(name)
        except Exception:
            continue
        for fn in ("knn", "get_graph_feature"):
            rebind(mod, fn, getattr(dgcnn_util, fn), name)
    try:  # the encoder's forward: fused EdgeConv layers where a block qualifies, the reference's own sequence otherwise
        enc = None if not edgeconv else getattr(importlib.import_module("models.dgcnn_util"), "dgcnn_encoder", None)
        if enc is not None and enc.forward is not dgcnn_util.dgcnn_encoder_forward:
            enc.forward = dgcnn_util.dgcnn_encoder_forward
            patched.append("models.dgcnn_util.dgcnn_encoder.forward")
    except Exception:
        pass
    # the patch Encoder (mini-PointNet) of every transformer model that defines one: forward on the tensor cores
    if edgeconv:
        from . import encoder
        for mname, mod in list(sys.modules.items()):
            if mod is None or not mname.startswith("models."):
                continue
            cls = vars(mod).get("Encoder")
            if isinstance(cls, type) and getattr(cls, "__module__", None) == mname and hasattr(cls, "forward") \
                    and cls.forward is not encoder.encoder_forward:
                cls._pdae_reference_forward = cls.forward
                cls.forward = encoder.encoder_forward
                patched.append(mname + ".Encoder.forward")
    try:
        rebind(importlib.import_module("utils.misc"), "fps", group.fps, "utils.misc")
    except Exception:
        pass
    try:  # corruptions run inside forward: Drop-Patch (datasets/corrupt_util_tensor.py:592-616) and the affine chain
        cut = importlib.import_module("datasets.corrupt_util_tensor")  # (:59-343, :706-728), one launch per chain
        for fn in ("dropout_patch_random", "corrupt_data", "corrupt_scale_nonorm", "corrupt_tranlate", "corrupt_rotate_360",
                   "corrupt_rotate_z_360", "corrupt_reflection", "corrupt_shear"):
            rebind(cut, fn, getattr(corrupt_util_tensor, fn), "datasets.corrupt_util_tensor")
        cut.corruptions.update(corrupt_util_tensor.corruptions)
    except Exception:
        pass
    # every flavour of the patchifier class the reference defines, by the module that defines it
    flavours = {"models.PointCAE_transformer": group.Group, "models.Point_MAE": group.Group,
                "models.Point_MlMAE": group.Group, "models.PointCAE_pointnetv2": group.Group,
                "models.Point_M2AE_modules": group.GroupWithIndex, "models.MaskSurf": group.GroupNormal,
                "models.MaskSurf_v2": group.GroupAttribute, "models.MaskFeat_transformer": group.GroupAttribute,
                "models.MaskFeat_DGCNN": group.GroupAttribute}
    for name, cls in flavours.items():
        mod = sys.modules.get(name)
        if mod is not None:
            rebind(mod, "Group", cls, name)
    # the same objects under other names: modules that imported them from the defining module
    for mname, mod in list(sys.modules.items()):
        if mod is None or mname.split(".")[0] not in ("models", "datasets", "utils", "tools", "segmentation"):
            continue
        for attr, val in list(vars(mod).items()):
            hit = replaced.get(id(val))
            if hit is not None and hit[0] is val:
                setattr(mod, attr, hit[1])
                patched.append(mname + "." + attr)
    return patched
