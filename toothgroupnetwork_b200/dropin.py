"""Make the reference's import paths resolve to this package.

    import toothgroupnetwork_b200.dropin as dropin
    dropin.install()
    from models.modules import pointnet_pp        # reference code, unmodified

After ``install()`` the modules the reference's callers import
(``blocks.py:6``, ``heads.py:6``, ``basic_operators.py:4``, ``gen_utils.py:8``, ``pointnet_pp.py:3``,
``tsg_centroid_module.py:3``, ``tsg_seg_module.py:3``, ``tsegnet.py:8``, ``tgn_loss.py:4``,
``tsg_loss.py:2`` ...) are served from here:

    external_libs.pointops.functions.pointops      -> toothgroupnetwork_b200.pointops
    external_libs.pointnet2_utils.pointnet2_utils  -> toothgroupnetwork_b200.pointnet2_utils
    pointops_cuda                                  -> toothgroupnetwork_b200.pointops_cuda

Existing ``external_libs`` packages on ``sys.path`` (the reference checkout) keep serving every
other submodule (``external_libs.scheduler`` ...): only the three names above are overridden.
"""
from __future__ import annotations

import importlib
import sys
import types

_TARGETS = {
    "external_libs.pointops.functions.pointops": "toothgroupnetwork_b200.pointops",
    "external_libs.pointnet2_utils.pointnet2_utils": "toothgroupnetwork_b200.pointnet2_utils",
    "pointops_cuda": "toothgroupnetwork_b200.pointops_cuda",
}


def _ensure_package(name: str) -> types.ModuleType:
    if name in sys.modules:
        return sys.modules[name]
    try:
        return importlib.import_module(name)
    except Exception:
        pkg = types.ModuleType(name)
        pkg.__path__ = []          # namespace-like package
        sys.modules[name] = pkg
        if "." in name:
            parent, _, child = name.rpartition(".")
            setattr(_ensure_package(parent), child, pkg)
        return pkg


def install() -> None:
    for alias, target in _TARGETS.items():
        mod = importlib.import_module(target)
        if "." in alias:
            parent, _, child = alias.rpartition(".")
            setattr(_ensure_package(parent), child, mod)
        sys.modules[alias] = mod


def accelerate_ops_utils(ops_utils_module=None) -> None:
    """Optional: also replace the host-side crop search of the reference's ``ops_utils`` (sklearn KDTree.query(k=3072),
    ops_utils.py:146-161, and the gather :198-218) with the GPU versions of ``toothgroupnetwork_b200.crops``.  Call after
    ``install()``; imports ``ops_utils`` from ``sys.path`` when no module is passed."""
    from . import clustering, crops
    if ops_utils_module is None:
        ops_utils_module = importlib.import_module("ops_utils")
    crops.accelerate(ops_utils_module)
    clustering.accelerate(ops_utils_module)        # DBSCAN + noise vote of get_clustering_labels (ops_utils.py:86-144)
    for name in ("models.modules.tsegnet", "inference_pipelines.inference_pipeline_tsegnet"):
        if name in sys.modules:                     # their own ``from sklearn.cluster import DBSCAN`` (tsegnet.py:7,59)
            clustering.accelerate_dbscan(sys.modules[name])


def accelerate_blocks(blocks_module=None) -> None:
    """Optional: run the no-grad forwards of the reference's ``PointTransformerLayer`` / ``TransitionDown``
    (models/modules/cbl_point_transformer/blocks.py:31-44, :59-79) on the fused kernels of
    ``toothgroupnetwork_b200.blocks_fused``; under autograd the reference's own code keeps running."""
    from . import blocks_fused
    if blocks_module is None:
        blocks_module = importlib.import_module("models.modules.cbl_point_transformer.blocks")
    blocks_fused.accelerate(blocks_module)


def accelerate_inference_tgn(module=None) -> None:
    """Optional: run the boundary stage of the reference's tgnet inference pipeline on the GPU -- its
    ``InferencePipeLine.get_boundary_sampled_feats`` (inference_pipeline_tgn.py:289-330: KDTree k = 40 label vote,
    uniform + FPS resampling) and the module's other ``KDTree`` searches (:107-140), see
    ``toothgroupnetwork_b200.boundary``.  Imports ``inference_pipelines.inference_pipeline_tgn`` from ``sys.path`` when
    no module is passed."""
    from . import boundary
    if module is None:
        module = importlib.import_module("inference_pipelines.inference_pipeline_tgn")
    boundary.accelerate_inference_pipeline(module)


def uninstall() -> None:
    for alias in _TARGETS:
        sys.modules.pop(alias, None)
