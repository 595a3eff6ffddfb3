"""Restatements of the tgnet boundary stage for the tests (TEST INFRASTRUCTURE ONLY; never imported by
toothgroupnetwork_b200/), and the seeded inputs its fixtures are made from.

* ``knn_f64``: the k nearest points by a float64 brute force, ``lexsort((index, rdist))`` with scikit-learn's
  ``rdist = (dx*dx + dy*dy) + dz*dz``, in query chunks.
* ``count_unique_by_row``: gen_utils.py:26-32, restated.
* ``boundary_sampled_feats``: ``InferencePipeLine.get_boundary_sampled_feats`` (inference_pipeline_tgn.py:289-330) in
  numpy, with the FPS of ``gen_utils.fps`` served by the oracle's C restatement of the reference kernel.
* ``boundary_case``: the seeded inputs of tests/golden/ref_boundary_sampling.npz.
"""
from __future__ import annotations

import os
import sys
from typing import Dict, Tuple

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# the reference's boundary_sampling_info (inference_pipeline_maker.py:56-60)
BOUNDARY_INFO = {"bdl_ratio": 0.7, "num_of_bdl_points": 20000, "num_of_all_points": 24000}

# name -> (raw vertices, sampled points, arch seed, subset seed, labelled)
CASES: Dict[str, Tuple[int, int, int, int, bool]] = {
    "v30k": (30000, 24000, 31, 131, True),
    "v100k": (100000, 24000, 32, 132, True),
    "v200k": (200000, 24000, 33, 133, True),
    "v24k_no_boundary": (24000, 24000, 34, 134, False),      # one label everywhere: no boundary row, FPS refuses
}
SEEDS = {"v30k": 7, "v100k": 8, "v200k": 9, "v24k_no_boundary": 10}    # np.random.seed before the call


def rdist(points: np.ndarray, q: np.ndarray) -> np.ndarray:
    d = points[None, :, :] - q[:, None, :]
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def knn_f64(points, queries, k: int, chunk: int = 256) -> Tuple[np.ndarray, np.ndarray]:
    """(dist (m,k) float64, idx (m,k) int64): ascending (rdist, index), dist = sqrt(rdist)."""
    p = np.asarray(points, np.float64)
    q = np.asarray(queries, np.float64)
    idx = np.empty((q.shape[0], k), np.int64)
    dist = np.empty((q.shape[0], k), np.float64)
    ar = np.arange(p.shape[0])
    for s in range(0, q.shape[0], chunk):
        d = rdist(p, q[s:s + chunk])
        part = np.argpartition(d, k - 1, axis=1)[:, :k] if k < p.shape[0] else np.broadcast_to(ar, d.shape)
        kth = np.take_along_axis(d, part, 1).max(1, keepdims=True)
        for r in range(d.shape[0]):                       # every point at or below the k-th rdist, then exact order
            cand = np.nonzero(d[r] <= kth[r])[0]
            order = np.lexsort((cand, d[r, cand]))[:k]
            idx[s + r] = cand[order]
            dist[s + r] = np.sqrt(d[r, cand[order]])
    return dist, idx


def count_unique_by_row(a: np.ndarray) -> np.ndarray:
    """gen_utils.count_unique_by_row: every first occurrence of a value in a row holds that value's count in the row."""
    weight = 1j * np.linspace(0, a.shape[1], a.shape[0], endpoint=False)
    b = a + weight[:, np.newaxis]
    _, ind, cnt = np.unique(b, return_index=True, return_counts=True)
    out = np.zeros_like(a)
    np.put(out, ind, cnt)
    return out


def _fps(xyz: np.ndarray, npoint: int) -> np.ndarray:
    from oracle import oracle as O
    if xyz.shape[0] <= npoint:
        raise TypeError("exceptions must derive from BaseException")      # gen_utils.fps: raise "new fps error"
    x = np.ascontiguousarray(np.asarray(xyz, np.float64).astype(np.float32))
    return O.furthestsampling(x, np.array([x.shape[0]], np.int32), np.array([npoint], np.int32)).astype(np.int64)


def boundary_sampled_feats(point_labels, org_feats, sampled_feats, bdl_ratio=0.7, num_of_bdl_points=20000, num_of_all_points=24000,
                           k: int = 40):
    """inference_pipeline_tgn.py:289-330 restated (sample_output_features None)."""
    _, near = knn_f64(sampled_feats[:, :3], org_feats[:, :3], k)
    counts = count_unique_by_row(point_labels[near])
    bd = counts[:, 0] / float(k) < bdl_ratio
    ps = point_labels[near[:, 0]].reshape(-1, 1)
    perm = np.random.permutation(int(bd.sum()))
    bd_feat, bd_lab = org_feats[bd][perm[:num_of_bdl_points]], ps[bd][perm[:num_of_bdl_points]]
    npoint = num_of_all_points - bd_feat.shape[0]
    f = _fps(org_feats[~bd][:, :3], npoint)
    non_feat, non_lab = org_feats[~bd][f[:npoint]], ps[~bd][f[:npoint]]
    return (np.concatenate([bd_feat, non_feat], 0), np.concatenate([bd_lab, non_lab], 0), bd_feat, bd_lab)


def boundary_case(name: str):
    """(point_labels (N',) float64, org_feats (N,6) float64, sampled_feats (N',6) float64) of a fixture case: a seeded
    dental arch (xyz + normals), a torch-seeded subset of N' vertices as the sampled points, and per-point labels tooth bin
    + 1 (gingiva 0) -- or 0 everywhere for the no-boundary case.  numpy's global RNG is not touched."""
    from toothgroupnetwork_b200 import clouds
    n, n_s, seed, sub_seed, labelled = CASES[name]
    xyz, normal, label = clouds.dental_arch(n, seed)
    org = torch.cat([xyz, normal], 1).double().numpy()
    sel = torch.randperm(n, generator=torch.Generator().manual_seed(sub_seed))[:n_s].numpy()
    sampled = org[sel].copy()
    lab = (label[torch.from_numpy(sel)] + 1).double().numpy() if labelled else np.zeros(n_s, np.float64)
    return lab, org, sampled
