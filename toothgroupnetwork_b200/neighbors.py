"""Exact float64 k-nearest-neighbour search with scikit-learn ``KDTree`` semantics, on the GPU.

The tgnet inference pipeline asks a host ``KDTree`` for neighbours on float64 arrays: k = 40 and k = 1 of every raw-mesh
vertex among the 24 000 sampled points (the boundary step, ``inference_pipeline_tgn.py:289-330``), k = 1 for the boundary
clusters and for the final label transfer (:107-140), and training repeats the k = 40 search
(``bdl_grouping_netowrk_model.py:146-161``).  Here one CUDA kernel (csrc/knn_f64.cu) answers them with the tree's
arithmetic: ``rdist = (dx*dx + dy*dy) + dz*dz`` in float64 without FMA contraction, results in ascending
``(rdist, index)`` order, distances ``sqrt(rdist)`` correctly rounded.  Where no two candidates tie that is exactly what
``KDTree.query`` returns; exact ties come out lower index first (the tree's own order among ties depends on its traversal).

* ``knn_f64(points, queries, k, return_distance=False)`` -- device tensors in and out.
* ``Grid`` -- the grid over one point set, built once and queried any number of times (also the fused label vote of the
  boundary step, see ``Grid.label_vote``).
* ``KDTree`` -- the slice of ``sklearn.neighbors.KDTree`` the reference uses: numpy in, numpy out; CUDA tensors in, CUDA
  tensors out.

k is limited to 64 (the crop searches with k = 3072 live in ``crops``).  There is no CPU path: without CUDA every entry
point raises ``TgnError``.
"""
from __future__ import annotations

from typing import Tuple, Union

import numpy as np
import torch

from . import _lib as L

MAX_K = 64


def _require_device() -> None:
    if not torch.cuda.is_available():
        raise L.TgnError("toothgroupnetwork_b200.neighbors needs a CUDA device (no CPU path)")


def _as_xyz(x: torch.Tensor, what: str) -> torch.Tensor:
    L.require_cuda(x)
    if x.dim() != 2 or x.shape[1] != 3:
        raise L.TgnError(f"{what}: expected an (n, 3) array, got shape {tuple(x.shape)}")
    return x.to(torch.float64).contiguous()          # float32 -> float64 is exact


class Grid:
    """The uniform grid of csrc/knn_f64.cu over one float64 point set (n, 3) on the device."""

    def __init__(self, points: torch.Tensor):
        _require_device()
        self.points = _as_xyz(points, "points")
        self.n = int(self.points.shape[0])
        if self.n == 0:
            raise ValueError("the point set is empty")
        lib = L.load()
        self.workspace = torch.empty(int(lib.tgn_knn_f64_bytes(self.n)), dtype=torch.uint8, device=self.points.device)
        L.call("tgn_knn_f64_build", self.n, L.ptr(self.points), L.ptr(self.workspace), L.stream_ptr())

    def _check(self, queries: torch.Tensor, k: int) -> torch.Tensor:
        q = _as_xyz(queries.to(self.points.device), "queries")
        if k > MAX_K:
            raise L.TgnError(f"k={k} exceeds {MAX_K} (knn_f64 keeps the k best in registers)")
        if k > self.n:
            raise ValueError("k must be less than or equal to the number of training points")
        if k < 1:
            raise ValueError(f"k must be at least 1, got {k}")
        return q

    def query(self, queries: torch.Tensor, k: int, return_distance: bool = False):
        """idx (m, k) int64 of the k nearest points of every query, ascending (rdist, index); with ``return_distance``
        ``(dist (m, k) float64, idx)``."""
        q = self._check(queries, int(k))
        m = int(q.shape[0])
        idx = torch.empty((m, k), dtype=torch.int64, device=q.device)
        dist = torch.empty((m, k), dtype=torch.float64, device=q.device) if return_distance else None
        L.call("tgn_knn_f64_query", self.n, m, int(k), L.ptr(q), L.ptr(self.workspace), L.ptr(idx), L.ptr(dist),
               None, 0.0, None, None, None, L.stream_ptr())
        return (dist, idx) if return_distance else idx

    def label_vote(self, queries: torch.Tensor, labels: torch.Tensor, k: int, ratio: float
                   ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        """For every query: the label of its nearest point (float64), whether fewer than ``ratio`` of its k nearest points
        carry that label (bool, ``count / k < ratio`` evaluated in float64), and the number of such queries (int32 (1,),
        on the device).  ``count_unique_by_row(labels[idx])[:, 0] / k < ratio`` without the (m, k) index matrix."""
        q = self._check(queries, int(k))
        lab = labels.to(q.device).reshape(-1).to(torch.float64).contiguous()
        if lab.shape[0] != self.n:
            raise L.TgnError(f"labels: expected {self.n} values, got {lab.shape[0]}")
        m = int(q.shape[0])
        nearest = torch.empty((m,), dtype=torch.float64, device=q.device)
        is_bd = torch.empty((m,), dtype=torch.bool, device=q.device)
        count = torch.empty((1,), dtype=torch.int32, device=q.device)
        L.call("tgn_knn_f64_query", self.n, m, int(k), L.ptr(q), L.ptr(self.workspace), None, None,
               L.ptr(lab), float(ratio), L.ptr(nearest), L.ptr(is_bd), L.ptr(count), L.stream_ptr())
        return nearest, is_bd, count


def knn_f64(points: torch.Tensor, queries: torch.Tensor, k: int, return_distance: bool = False):
    """The k <= 64 nearest ``points`` (n, 3) of every row of ``queries`` (m, 3), CUDA tensors, float32 or float64:
    idx (m, k) int64 in ascending (rdist, index) order, or ``(dist float64, idx)`` with ``return_distance``."""
    return Grid(points).query(queries, k, return_distance)


_EUCLIDEAN = ("euclidean", "l2")


class KDTree:
    """Stand-in for ``sklearn.neighbors.KDTree`` as the reference uses it (``KDTree(X, leaf_size=...)`` then
    ``.query(X, k, return_distance)``), served by ``Grid``.  ``leaf_size`` is accepted and ignored."""

    def __init__(self, X, leaf_size: int = 40, metric: str = "minkowski", **kwargs):
        p = kwargs.pop("p", 2)
        if not (metric in _EUCLIDEAN or (metric == "minkowski" and p == 2)):
            raise L.TgnError(f"KDTree: only the euclidean metric is implemented (got metric={metric!r}, p={p})")
        if kwargs:
            raise L.TgnError(f"KDTree: unsupported options {sorted(kwargs)}")
        _require_device()
        if torch.is_tensor(X):
            pts = X
        else:
            a = np.asarray(X, dtype=np.float64)
            if a.ndim != 2:
                raise ValueError(f"Expected 2D array, got {a.ndim}D array instead")
            pts = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        if pts.dim() != 2 or pts.shape[0] == 0:
            raise ValueError(f"Found array with shape {tuple(pts.shape)}: KDTree needs at least one sample")
        self.leaf_size = leaf_size
        self._grid = Grid(pts)

    def query(self, X, k: int = 1, return_distance: bool = True, dualtree: bool = False, breadth_first: bool = False,
              sort_results: bool = True) -> Union[np.ndarray, torch.Tensor, Tuple]:
        """``(dist float64 (m, k), ind int64 (m, k))``, or ``ind`` alone; sorted ascending whatever ``sort_results`` says
        (an unsorted answer is any order, this one included)."""
        as_numpy = not torch.is_tensor(X)
        if as_numpy:
            a = np.asarray(X, dtype=np.float64)
            if a.ndim != 2:
                raise ValueError(f"Expected 2D array, got {a.ndim}D array instead")
            if a.shape[0] == 0:
                raise ValueError(f"Found array with 0 sample(s) (shape={a.shape}) while a minimum of 1 is required.")
            if a.shape[1] != 3:
                raise ValueError("query data dimension must match training data dimension")
            q = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        else:
            q = X
            if q.dim() != 2 or q.shape[0] == 0:
                raise ValueError(f"Found array with shape {tuple(q.shape)} while a minimum of 1 sample is required.")
        k = int(k)
        if k > self._grid.n:
            raise ValueError("k must be less than or equal to the number of training points")
        out = self._grid.query(q, k, return_distance)
        if not as_numpy:
            return out
        if return_distance:
            return out[0].cpu().numpy(), out[1].cpu().numpy()
        return out.cpu().numpy()
