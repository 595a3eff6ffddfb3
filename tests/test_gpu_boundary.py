"""GPU: the float64 kNN (csrc/knn_f64.cu, toothgroupnetwork_b200/neighbors.py) against a float64 brute force and
scikit-learn's KDTree, its fused label vote against count_unique_by_row, and the boundary stage
(toothgroupnetwork_b200/boundary.py) against the reference's own method: the stored fixture, and live where the reference
checkout is staged."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import boundary_oracle as B  # noqa: E402
from oracle import golden, ref_models  # noqa: E402
from toothgroupnetwork_b200 import _lib, boundary, clouds, neighbors  # noqa: E402

pytestmark = pytest.mark.gpu

GOLD = golden.Golden("ref_boundary_sampling", record=False)
OUT_KEYS = ("results_feat", "results_label", "bd_feat", "bd_label")


def check_knn(points: np.ndarray, queries: np.ndarray, k: int, dtype=torch.float64):
    wd, wi = B.knn_f64(points.astype(np.float64), queries.astype(np.float64), k)
    p, q = torch.from_numpy(points).to(dtype).cuda(), torch.from_numpy(queries).to(dtype).cuda()
    gd, gi = neighbors.knn_f64(p, q, k, return_distance=True)
    assert gi.dtype == torch.int64 and gd.dtype == torch.float64
    gi, gd = gi.cpu().numpy(), gd.cpu().numpy()
    assert np.array_equal(gi, wi), f"k={k}: {int((gi != wi).any(1).sum())} rows differ"
    assert gd.tobytes() == wd.tobytes()
    assert np.array_equal(neighbors.knn_f64(p, q, k).cpu().numpy(), wi)


@pytest.mark.parametrize("k", [1, 3, 10, 40, 64])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_knn_f64_matches_bruteforce_on_an_arch(k, dtype):
    xyz, _, _ = clouds.dental_arch(12000, 3)
    pts = xyz.numpy() if dtype == torch.float32 else xyz.double().numpy() + np.random.default_rng(0).normal(size=(12000, 3)) * 1e-4
    q_xyz, _, _ = clouds.dental_arch(3000, 4)
    q = np.concatenate([q_xyz.double().numpy(), [[0.0, 0.0, 0.0], [1.5, -2.0, 0.7], [-40.0, 25.0, 90.0], [1e6, 0.0, -1e6]]])
    if dtype == torch.float32:
        q = q.astype(np.float32)
    check_knn(pts, q, k, dtype)


@pytest.mark.parametrize("k", [1, 40, 64])
def test_knn_f64_small_sets_duplicates_and_n_equal_k(k):
    rng = np.random.default_rng(k)
    check_knn(rng.normal(size=(k, 3)), rng.normal(size=(50, 3)) * 3, k)                       # n == k
    check_knn(rng.normal(size=(k + 5, 3)) * [1, 1e-3, 0], rng.normal(size=(40, 3)), k)        # < 2 cells on some axes
    dup = clouds.with_duplicates(clouds.cube(2000, 5), 6).double().numpy()                    # every point twice: exact ties
    check_knn(dup, np.concatenate([dup[:300], clouds.cube(200, 7).double().numpy()]), k)
    check_knn(np.zeros((70, 3)), np.array([[0.0, 0.0, 0.0], [1.0, 2.0, 3.0]]), k)              # all points identical


def test_kdtree_matches_sklearn_on_an_arch():
    from sklearn.neighbors import KDTree
    xyz, normal, _ = clouds.dental_arch(100000, 21)
    org = xyz.double().numpy()
    sampled = org[torch.randperm(100000, generator=torch.Generator().manual_seed(22))[:24000].numpy()].copy()
    ref, ours = KDTree(sampled, leaf_size=40), neighbors.KDTree(sampled, leaf_size=40)
    for k in (1, 40):
        wd, wi = ref.query(org, k=k)
        gd, gi = ours.query(org, k=k)
        assert isinstance(gi, np.ndarray) and np.array_equal(gi, wi), k
        assert gd.tobytes() == wd.tobytes(), k
        assert np.array_equal(ours.query(org, k=k, return_distance=False), wi)
    gi_t = ours.query(torch.from_numpy(org).cuda(), k=1, return_distance=False)
    assert gi_t.is_cuda and np.array_equal(gi_t.cpu().numpy(), ref.query(org, k=1, return_distance=False))
    with pytest.raises(ValueError, match="k must be less than or equal to the number of training points"):
        neighbors.KDTree(sampled[:10]).query(org[:5], k=11)
    with pytest.raises(ValueError):
        ours.query(np.zeros((0, 3)), k=1)
    with pytest.raises(_lib.TgnError):
        ours.query(org[:5], k=65)


def test_label_vote_matches_count_unique_by_row():
    xyz, _, label = clouds.dental_arch(24000, 41)
    pts = xyz.double().numpy()
    labels = (label + 1).double().numpy()
    # a query whose 40 nearest are 28 of one label and 12 of another: 28/40 == 0.7 is not a boundary
    labels_t = labels.copy()
    q_extra = np.array([[5.0, 5.0, 5.0]])
    pts = np.concatenate([pts, q_extra + np.arange(40)[:, None] * np.array([[1e-3, 0, 0]])])
    labels_t = np.concatenate([labels_t, np.r_[np.full(28, 3.0), np.full(12, 4.0)]])
    q_xyz, _, _ = clouds.dental_arch(20000, 42)
    q = np.concatenate([q_xyz.double().numpy(), q_extra, q_extra + [[0.039, 0, 0]]])
    _, near = B.knn_f64(pts, q, 40)
    counts = B.count_unique_by_row(labels_t[near])
    want_bd = counts[:, 0] / 40. < 0.7
    assert not want_bd[-2] and want_bd[-1]                     # 28 of 40 (not a boundary), and the far end: 12 of 40
    grid = neighbors.Grid(torch.from_numpy(pts).cuda())
    nl, bd, cnt = grid.label_vote(torch.from_numpy(q).cuda(), torch.from_numpy(labels_t).cuda(), 40, 0.7)
    assert np.array_equal(nl.cpu().numpy(), labels_t[near[:, 0]])
    assert np.array_equal(bd.cpu().numpy(), want_bd)
    assert int(cnt.item()) == int(want_bd.sum()) and 0 < int(want_bd.sum()) < q.shape[0]


def compare_with_fixture(name, got, post):
    fix = GOLD._load()
    if f"{name}.raises" in fix.files:
        raise AssertionError(f"{name}: the reference raised, this returned")
    for key, a in zip(OUT_KEYS, got):
        assert GOLD.exact(f"{name}.{key}", a, None), (name, key, GOLD.mismatch(f"{name}.{key}", a))
    assert post == float(fix[f"{name}.post_random"])


class Pipe:
    config = {"boundary_sampling_info": dict(B.BOUNDARY_INFO)}


@pytest.mark.parametrize("name", list(B.CASES))
def test_boundary_sampled_feats_matches_the_reference_fixture(name):
    labels, org, sampled = B.boundary_case(name)
    fix = GOLD._load()
    _, bd, cnt = neighbors.Grid(torch.from_numpy(sampled[:, :3].copy()).cuda()).label_vote(
        torch.from_numpy(org[:, :3].copy()).cuda(), torch.from_numpy(labels).cuda(), 40, 0.7)
    assert int(cnt.item()) == int(fix[f"{name}.n_bd"]) == int(bd.sum())
    np.random.seed(B.SEEDS[name])
    if f"{name}.raises" in fix.files:
        with pytest.raises(TypeError):
            boundary.get_boundary_sampled_feats(Pipe(), labels, org, sampled, None)
        assert np.random.random() == float(fix[f"{name}.post_random"])
        return
    got = boundary.get_boundary_sampled_feats(Pipe(), labels, org, sampled, None)
    compare_with_fixture(name, got, np.random.random())


@pytest.mark.parametrize("name", ["v30k", "v200k"])
def test_boundary_sampled_feats_matches_the_reference_live(name):
    """The reference's own method in World("reference") (its FPS the verbatim reference kernel) against the accelerated
    class, same numpy seed on both sides."""
    if not ref_models.available():
        pytest.skip("reference checkout not staged")
    labels, org, sampled = B.boundary_case(name)
    world = ref_models.World("reference")
    try:
        with world:
            tgn = importlib.import_module("inference_pipelines.inference_pipeline_tgn")
            pipe = tgn.InferencePipeLine.__new__(tgn.InferencePipeLine)
            pipe.config = {"boundary_sampling_info": dict(B.BOUNDARY_INFO)}
            np.random.seed(B.SEEDS[name])
            want = pipe.get_boundary_sampled_feats(labels, org, sampled, None)
            want_post = np.random.random()
            boundary.accelerate_inference_pipeline(tgn)
            np.random.seed(B.SEEDS[name])
            got = pipe.get_boundary_sampled_feats(labels, org, sampled, None)
            got_post = np.random.random()
            assert tgn.KDTree is neighbors.KDTree
    finally:
        for mod in list(sys.modules):
            if mod.split(".")[0] == "inference_pipelines":
                del sys.modules[mod]
    for key, w, g in zip(OUT_KEYS, want, got):
        assert g.dtype == w.dtype and g.shape == w.shape and g.tobytes() == w.tobytes(), key
    assert got_post == want_post
    compare_with_fixture(name, got, got_post)
