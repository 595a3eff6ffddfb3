"""DBSCAN / get_clustering_labels on the device against scikit-learn (the reference's own dependency, ops_utils.py:86-144)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import golden  # noqa: E402
from toothgroupnetwork_b200 import clouds, clustering  # noqa: E402

pytestmark = pytest.mark.gpu
sklearn_cluster = pytest.importorskip("sklearn.cluster")
G = golden.Golden("ref_live_clustering")      # the reference's get_clustering_labels results (oracle/golden.py)


def moved_cloud(n, seed, pull, jitter):
    """points pulled towards their tooth centroid like the offsets of a (partly) trained network"""
    xyz, _, label = clouds.dental_arch(n, seed)
    xyz, label = xyz.numpy(), label.numpy().astype(np.int64)
    label = np.where(label < 0, 0, label)
    cent = np.stack([xyz[label == c].mean(0) if (label == c).any() else np.zeros(3, np.float32) for c in range(int(label.max()) + 1)])
    rng = np.random.default_rng(seed)
    moved = xyz + pull * (cent[label] - xyz) + rng.normal(0, jitter, xyz.shape)
    return moved.astype(np.float32), label


def check_against_sklearn(pts, eps=0.03, min_samples=30):
    ref = sklearn_cluster.DBSCAN(eps=eps, min_samples=min_samples).fit(pts)
    labels, core = clustering.dbscan(pts, eps, min_samples)
    assert labels.dtype == ref.labels_.dtype
    assert np.array_equal(core, ref.core_sample_indices_)
    assert np.array_equal(labels, ref.labels_)
    return ref


@pytest.mark.parametrize("n,pull,jitter", [(24000, 0.0, 0.0), (24000, 0.5, 0.004), (24000, 0.9, 0.004), (24000, 1.0, 0.0005), (6000, 0.7, 0.01), (997, 0.9, 0.002)])
def test_dbscan_equals_sklearn_on_moved_arches(n, pull, jitter):
    pts, label = moved_cloud(n, 1, pull, jitter)
    ref = check_against_sklearn(pts[label != 0])
    assert len(ref.labels_) > 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_dbscan_equals_sklearn_with_noise_borders_and_duplicates(seed):
    rng = np.random.default_rng(seed)
    blobs = [rng.normal(c, s, (m, 3)) for c, s, m in ((0.0, 0.02, 900), (0.3, 0.01, 400), (-0.4, 0.05, 1500), (0.8, 0.004, 40))]
    pts = np.concatenate(blobs + [rng.uniform(-1, 1, (3000, 3))]).astype(np.float32)
    pts = np.concatenate([pts, pts[:200]])                           # exact duplicates
    pts = pts[rng.permutation(len(pts))]
    ref = check_against_sklearn(pts)
    assert (ref.labels_ == -1).any() and (ref.labels_ >= 0).any()
    # border points exist: labelled but not core
    assert ((ref.labels_ >= 0).sum() > len(ref.core_sample_indices_))
    check_against_sklearn(pts, eps=0.05, min_samples=5)
    check_against_sklearn(pts, eps=0.011, min_samples=3)


@pytest.mark.parametrize("name", ["blobs", "blobs_loose", "arch"])
def test_dbscan_equals_the_sklearn_fixture_and_the_oracle(name):
    """no scikit-learn needed at run time: tests/golden/ref_sklearn_dbscan.npz + the oracle's restatement"""
    from oracle import oracle as O
    fix = np.load(os.path.join(ROOT, "tests", "golden", "ref_sklearn_dbscan.npz"))
    pts, eps, ms = fix[name + "_points"], float(fix[name + "_eps"]), int(fix[name + "_min_samples"])
    labels, core = clustering.dbscan(pts, eps, ms)
    assert np.array_equal(labels, fix[name + "_labels"]) and np.array_equal(core, fix[name + "_core"])
    o_labels, o_core = O.dbscan(pts, eps, ms)
    assert np.array_equal(labels, o_labels) and np.array_equal(core, o_core)


def test_dbscan_small_and_degenerate_inputs():
    for pts in (np.zeros((0, 3), np.float32), np.zeros((1, 3), np.float32), np.zeros((40, 3), np.float32),
                np.linspace(0, 100, 90, dtype=np.float32).reshape(30, 3)):
        if len(pts) == 0:
            labels, core = clustering.dbscan(pts)
            assert labels.shape == (0,) and core.shape == (0,)
        else:
            check_against_sklearn(pts)
    wide = np.random.default_rng(0).uniform(-50, 50, (20000, 3)).astype(np.float32)       # cells wider than eps
    check_against_sklearn(wide, eps=2.0, min_samples=4)


@pytest.mark.parametrize("n,pull,jitter,outliers", [(8000, 0.0, 0.0, 0.0), (16000, 0.0, 0.0, 0.0), (24000, 0.6, 0.004, 0.01), (24000, 0.93, 0.003, 0.03), (24000, 0.6, 0.004, 0.0)])
def test_get_clustering_labels_equals_the_reference_function(n, pull, jitter, outliers):
    """the whole of ops_utils.get_clustering_labels: DBSCAN, elongation test (+ MeanShift split), noise vote"""
    pts, label = moved_cloud(n, 2, pull, jitter)
    rng = np.random.default_rng(3)
    label = label.copy()
    label[rng.random(len(label)) < 0.02] = 0                         # holes in the foreground
    stray = rng.random(len(pts)) < outliers                          # predictions that went astray: DBSCAN noise
    pts[stray] += rng.normal(0, 0.08, (int(stray.sum()), 3)).astype(np.float32)

    def reference():                                                 # the labels, or the name of the error the reference raises
        from oracle import ref_models
        w = ref_models.World("reference")
        try:
            with w:
                return w.mod("ops_utils").get_clustering_labels(pts.copy(), label.copy())
        except (IndexError, ValueError) as e:
            return np.asarray(type(e).__name__)
    want = G.array(f"labels_{n}_{pull}_{jitter}_{outliers}", reference)
    try:
        got = clustering.get_clustering_labels(pts, label)
    except (IndexError, ValueError) as e:                            # fewer than three clusters: the reference's own IndexError (:124-126)
        assert want.dtype.kind == "U" and want.item() == type(e).__name__, want
        return
    if want.dtype.kind == "U":
        # the reference hands KDTree.query an empty array when DBSCAN leaves no noise (ops_utils.py:135) and raises; here the
        # vote is skipped and the DBSCAN labels are the answer
        assert want.item() == "ValueError"
        assert outliers == 0.0
        want = sklearn_cluster.DBSCAN(eps=0.03, min_samples=30).fit(pts[label != 0]).labels_
        assert (want != -1).all()
    assert got.dtype == want.dtype and np.array_equal(got, want)


def test_sklearn_shaped_class_on_the_other_call_sites():
    """tsegnet.py:59 (DBSCAN(eps=0.05, min_samples=3) over a few hundred moved centroid candidates) and
    ops_utils.clustering_points(method="dbscan") (:28, eps=0.03, min_samples=60)."""
    rng = np.random.default_rng(5)
    cand = np.concatenate([rng.normal(c, 0.01, (18, 3)) for c in rng.uniform(-0.5, 0.5, (14, 3))] + [rng.uniform(-0.6, 0.6, (20, 3))]).astype(np.float32)
    ref = sklearn_cluster.DBSCAN(eps=0.05, min_samples=3).fit(cand, 3)
    got = clustering.DBSCAN(eps=0.05, min_samples=3).fit(cand, 3)
    assert np.array_equal(got.labels_, ref.labels_) and np.array_equal(got.core_sample_indices_, ref.core_sample_indices_)
    assert np.array_equal(got.components_, ref.components_)
    assert np.array_equal(clustering.DBSCAN(eps=0.05, min_samples=3).fit_predict(cand), ref.labels_)
    from oracle import ref_models
    if ref_models.reference_root() is None:
        pytest.skip("reference checkout not staged")
    pts, label = moved_cloud(24000, 4, 0.9, 0.004)
    moved = [pts[label != 0], pts[label != 0][::2]]
    with ref_models.World("reference") as w:
        want = w.mod("ops_utils").clustering_points(moved, "dbscan")
    with ref_models.World("b200") as w:
        assert w.mod("ops_utils").DBSCAN is clustering.DBSCAN and w.mod("models.modules.tsegnet").DBSCAN is clustering.DBSCAN
        got = w.mod("ops_utils").clustering_points(moved, "dbscan")
    for a, b in zip(want, got):                                       # centroids, centroid labels, per-point labels
        for x, y in zip(a, b):
            assert np.array_equal(np.asarray(x), np.asarray(y))
