"""CPU: the oracle's restatements of the point-transformer blocks and of DBSCAN against fixtures made by the reference's own
Python (blocks.py imported from the reference checkout) and by scikit-learn (tests/golden/make_ref_blocks_golden.py); host-side
helpers of toothgroupnetwork_b200.clustering."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def _state(fix, tag):
    pre = tag + "_state_"
    return {k[len(pre):]: torch.from_numpy(fix[k]) for k in fix.files if k.startswith(pre)}


@pytest.mark.parametrize("c", [32, 64])
@pytest.mark.parametrize("train_bn", [True, False])
def test_oracle_point_transformer_layer_matches_the_reference_layer(c, train_bn):
    fix = np.load(os.path.join(GOLD, "ref_torch_blocks.npz"))
    tag = f"ptl{c}"
    p, o, x = torch.from_numpy(fix["p"]), torch.from_numpy(fix["o"]), torch.from_numpy(fix[tag + "_x"])
    want = torch.from_numpy(fix[tag + ("_out_train" if train_bn else "_out_eval")])
    got = O.point_transformer_layer(p, x, o, _state(fix, tag), int(fix[tag + "_K"]), 8, train_bn)
    assert got.shape == want.shape
    assert float((got - want).abs().max()) <= 2e-5 * float(want.abs().max())
    exact = O.point_transformer_layer(p, x, o, _state(fix, tag), int(fix[tag + "_K"]), 8, train_bn, dtype=torch.float64)
    assert float((exact.float() - want).abs().max()) <= 2e-5 * float(want.abs().max())


@pytest.mark.parametrize("train_bn", [True, False])
def test_oracle_transition_down_matches_the_reference_block(train_bn):
    fix = np.load(os.path.join(GOLD, "ref_torch_blocks.npz"))
    p, o, x = torch.from_numpy(fix["p"]), torch.from_numpy(fix["o"]), torch.from_numpy(fix["td_x"])
    n_p, n_x, n_o = O.transition_down(p, x, o, _state(fix, "td"), 4, 16, train_bn)
    assert np.array_equal(n_p.numpy(), fix["td_p"]) and np.array_equal(n_o.numpy(), fix["td_o"])
    want = torch.from_numpy(fix["td_out_train" if train_bn else "td_out_eval"])
    assert float((n_x - want).abs().max()) <= 2e-5 * float(want.abs().max())


@pytest.mark.parametrize("name", ["blobs", "blobs_loose", "arch"])
def test_oracle_dbscan_matches_sklearn_fixture(name):
    fix = np.load(os.path.join(GOLD, "ref_sklearn_dbscan.npz"))
    labels, core = O.dbscan(fix[name + "_points"], float(fix[name + "_eps"]), int(fix[name + "_min_samples"]))
    assert np.array_equal(core, fix[name + "_core"])
    assert np.array_equal(labels, fix[name + "_labels"])


def test_clustering_host_helpers():
    from toothgroupnetwork_b200 import clustering
    rows = np.array([[1, 1, 2, 2, 3], [5, 5, 5, 1, 1], [7, 8, 9, 9, 7], [104, 3, 104, 3, 0]])
    want = []
    for r in rows:                                                    # the reference's loop, ops_utils.py:139-141
        u, c = np.unique(r, return_counts=True)
        want.append(u[np.argmax(c)])
    assert np.array_equal(clustering._majority(rows), np.array(want))
    x = np.random.default_rng(0).normal(size=(400, 3)) * [3, 1, 0.2]
    from sklearn.decomposition import PCA
    assert np.allclose(clustering._explained_variance(x), PCA(n_components=3).fit(x).explained_variance_, rtol=1e-10)
    assert np.array_equal(clustering._explained_variance(x[:2]), np.array([0, 0, 0]))
    # float64 input is taken when it holds float32 values, refused otherwise (it would be clustered on rounded coordinates)
    f32 = np.random.default_rng(1).normal(size=(20, 3)).astype(np.float32)
    assert clustering._as_float32(f32.astype(np.float64)).dtype == np.float32
    with pytest.raises(clustering.L.TgnError):
        clustering._as_float32(f32.astype(np.float64) + 1e-12)


def test_dbscan_class_refuses_what_it_does_not_implement():
    from toothgroupnetwork_b200 import clustering
    with pytest.raises(clustering.L.TgnError):
        clustering.DBSCAN(eps=0.1, min_samples=3, metric="manhattan")
    with pytest.raises(clustering.L.TgnError):
        clustering.DBSCAN(eps=0.1, min_samples=3).fit(np.zeros((4, 2), np.float32))
    pts = np.zeros((4, 3), np.float32)
    if torch.cuda.is_available():                                    # the same call on a GPU runs there
        from sklearn.cluster import DBSCAN
        assert np.array_equal(clustering.DBSCAN(eps=0.1, min_samples=3).fit(pts).labels_, DBSCAN(eps=0.1, min_samples=3).fit(pts).labels_)
        return
    with pytest.raises(clustering.L.TgnError):                        # no CPU path: the product fails loudly without a GPU
        clustering.DBSCAN(eps=0.1, min_samples=3).fit(pts)
