"""CPU: the boundary-stage restatements (tests/boundary_oracle.py) against the reference's own method
(tests/golden/ref_boundary_sampling.npz, made by tests/golden/make_ref_boundary_golden.py) and against scikit-learn's
KDTree; the GPU-only entry points refuse to run without CUDA; the accelerator patches exactly two names."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import boundary_oracle as B  # noqa: E402
from oracle import golden  # noqa: E402

GOLD = golden.Golden("ref_boundary_sampling", record=False)
OUT_KEYS = ("results_feat", "results_label", "bd_feat", "bd_label")


def test_oracle_boundary_sampled_feats_matches_the_reference_method():
    name = "v30k"
    labels, org, sampled = B.boundary_case(name)
    np.random.seed(B.SEEDS[name])
    got = B.boundary_sampled_feats(labels, org, sampled, **B.BOUNDARY_INFO)
    post = np.random.random()
    for key, a in zip(OUT_KEYS, got):
        assert GOLD.exact(f"{name}.{key}", a, None), GOLD.mismatch(f"{name}.{key}", a)
    assert got[2].shape[0] == int(GOLD._load()[f"{name}.n_bd"])
    assert post == float(GOLD._load()[f"{name}.post_random"])


def test_oracle_knn_f64_matches_sklearn_kdtree():
    from sklearn.neighbors import KDTree
    rng = np.random.default_rng(5)
    pts = rng.normal(size=(3000, 3)) * [0.5, 0.3, 0.1]          # continuous float64: no two rdists tie
    q = np.concatenate([rng.normal(size=(400, 3)) * 0.4, [[4.0, -3.0, 2.0]]])
    tree = KDTree(pts, leaf_size=40)
    for k in (1, 7, 40, 64):
        wd, wi = tree.query(q, k=k)
        gd, gi = B.knn_f64(pts, q, k)
        assert np.array_equal(gi, wi) and gd.tobytes() == wd.tobytes(), k


def test_count_unique_by_row_restatement():
    a = np.array([[3, 3, 1, 3], [2, 1, 1, 2], [0, 5, 6, 7]], np.float64)
    c = B.count_unique_by_row(a)
    assert np.array_equal(c[:, 0], [3, 2, 1])


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the refusal without a CUDA device")
def test_neighbors_and_boundary_refuse_without_cuda():
    from toothgroupnetwork_b200 import _lib, boundary, neighbors
    pts = np.zeros((50, 3))
    with pytest.raises(_lib.TgnError):
        neighbors.KDTree(pts)
    with pytest.raises(_lib.TgnError):
        neighbors.knn_f64(torch.zeros(50, 3), torch.zeros(5, 3), 3)
    labels, org, sampled = np.zeros(50), np.zeros((80, 6)), np.zeros((50, 6))
    with pytest.raises(_lib.TgnError):
        boundary.boundary_sampled_feats(labels, org, sampled)


def test_kdtree_refuses_other_metrics():
    from toothgroupnetwork_b200 import _lib, neighbors
    with pytest.raises(_lib.TgnError):
        neighbors.KDTree(np.zeros((5, 3)), metric="manhattan")
    with pytest.raises(_lib.TgnError):
        neighbors.KDTree(np.zeros((5, 3)), metric="minkowski", p=1)


def test_boundary_refuses_sample_output_features():
    from toothgroupnetwork_b200 import _lib, boundary

    class Pipe:
        config = {"boundary_sampling_info": dict(B.BOUNDARY_INFO)}
    with pytest.raises(_lib.TgnError):
        boundary.get_boundary_sampled_feats(Pipe(), np.zeros(5), np.zeros((8, 6)), np.zeros((5, 6)), np.zeros((1, 4, 5)))


def test_accelerate_inference_pipeline_patches_two_names():
    from oracle import ref_models
    if not ref_models.available():
        pytest.skip("reference checkout not staged")
    from toothgroupnetwork_b200 import boundary, neighbors
    world = ref_models.World("reference", cpu_dry_run=True)
    try:
        with world:
            tgn = importlib.import_module("inference_pipelines.inference_pipeline_tgn")
        mod_before, cls_before = dict(vars(tgn)), dict(vars(tgn.InferencePipeLine))
        boundary.accelerate_inference_pipeline(tgn)
        mod_after, cls_after = dict(vars(tgn)), dict(vars(tgn.InferencePipeLine))
    finally:
        for name in list(sys.modules):
            if name.split(".")[0] == "inference_pipelines":
                del sys.modules[name]
    assert {k for k in mod_after if mod_after[k] is not mod_before.get(k)} == {"KDTree"}
    assert {k for k in cls_after if cls_after[k] is not cls_before.get(k)} == {"get_boundary_sampled_feats"}
    assert tgn.KDTree is neighbors.KDTree
    assert tgn.InferencePipeLine.get_boundary_sampled_feats is boundary.get_boundary_sampled_feats
