"""The boundary stage of the tgnet inference pipeline on the GPU.

After the first network, ``InferencePipeLine.get_boundary_sampled_feats`` (``inference_pipeline_tgn.py:289-330``) flags
the raw-mesh vertices near a label boundary and resamples the mesh around them for the second network.  The reference
does it on the host: a scikit-learn ``KDTree`` over the 24 000 sampled points, a k = 40 and a k = 1 query for every raw
vertex, a ``np.unique`` label count per row, then a uniform resample of the boundary vertices and an FPS of the rest.

Here the k = 40 search and the label count are one kernel (csrc/knn_f64.cu, exact float64 distances like the tree, the
label vote fused so no (n, 40) index matrix is written), the row selection and the FPS run on the device, and the
uniform resample draws ``np.random.permutation`` on the host exactly as ``gen_utils.resample_pcd`` does -- so the
result is bitwise the reference's for the same numpy seed, and numpy's global RNG is left in the same state (the
``KMeans(init="k-means++")`` of :270 draws from it next).  The only device->host synchronisation the output shapes need
is the read of the boundary count.

``accelerate_inference_pipeline(module)`` installs this method, and ``neighbors.KDTree`` for the module's other
``KDTree`` searches (:107, :114, :137-138), on an imported ``inference_pipelines.inference_pipeline_tgn``.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np
import torch

from . import _lib as L
from . import neighbors, pointops

K_BOUNDARY = 40            # neighbours counted per vertex (inference_pipeline_tgn.py:295-298)


def boundary_sampled_feats(point_labels, org_feats, sampled_feats, bdl_ratio: float = 0.7, num_of_bdl_points: int = 20000,
                           num_of_all_points: int = 24000) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """``(results_feat, results_label, bd_feat, bd_label)`` of the reference method for numpy inputs: ``point_labels``
    (N',) of the sampled points, ``org_feats`` (N, C) raw-mesh rows (xyz first), ``sampled_feats`` (N', >= 3)."""
    neighbors._require_device()
    lab_np = np.asarray(point_labels)
    org_np = np.ascontiguousarray(org_feats)
    dev = torch.device("cuda", torch.cuda.current_device())
    org = torch.from_numpy(org_np).to(dev)
    labels = torch.from_numpy(np.ascontiguousarray(lab_np, dtype=np.float64).reshape(-1)).to(dev)
    sampled = torch.from_numpy(np.ascontiguousarray(np.asarray(sampled_feats)[:, :3], dtype=np.float64)).to(dev)

    # k = 40 search + label vote; column 0 of the same search is the k = 1 query of :303
    nearest, is_bd, count = neighbors.Grid(sampled).label_vote(org[:, :3], labels, K_BOUNDARY, bdl_ratio)
    m = int(org.shape[0])
    n_bd = int(count.item())

    # boundary rows in order, resampled "uniformly" (gen_utils.resample_pcd :124-133): the same numpy draw as the reference
    bd_rows = torch.nonzero_static(is_bd, size=n_bd).reshape(-1)
    take = np.random.permutation(n_bd)[:num_of_bdl_points]
    bd_sel = bd_rows[torch.from_numpy(take).to(dev)]
    n_take = int(take.shape[0])

    # the other rows through FPS on their float32 xyz (gen_utils.fps :135-140, which refuses n <= npoint)
    npoint = int(num_of_all_points) - n_take
    n_non = m - n_bd
    if n_non <= npoint:
        raise TypeError(f"exceptions must derive from BaseException (new fps error: {n_non} points for {npoint} samples)")
    non_rows = torch.nonzero_static(~is_bd, size=n_non).reshape(-1)
    xyz32 = org[non_rows, :3].float().contiguous()
    offset = torch.tensor([n_non], dtype=torch.int32, device=dev)
    new_offset = torch.tensor([npoint], dtype=torch.int32, device=dev)
    fidx = pointops.fps_packed(xyz32, offset, new_offset, n_non, npoint)
    rows = torch.cat([bd_sel, non_rows[fidx.long()]])

    feats = org[rows].cpu().numpy()
    ps = nearest[rows].cpu().numpy().astype(lab_np.dtype, copy=False).reshape(-1, 1)
    return feats, ps, feats[:n_take].copy(), ps[:n_take].copy()


def get_boundary_sampled_feats(self, point_labels, org_feats, sampled_feats, sample_output_features):
    """Drop-in for ``InferencePipeLine.get_boundary_sampled_feats`` (inference_pipeline_tgn.py:289-330): reads
    ``self.config["boundary_sampling_info"]`` and returns the same four numpy arrays."""
    if sample_output_features is not None:
        raise L.TgnError("get_boundary_sampled_feats: sample_output_features is not implemented (the pipeline passes None)")
    info = self.config["boundary_sampling_info"]
    return boundary_sampled_feats(point_labels, org_feats, sampled_feats, float(info["bdl_ratio"]),
                                  int(info["num_of_bdl_points"]), int(info["num_of_all_points"]))


def accelerate_inference_pipeline(module) -> None:
    """Serve the boundary stage of an imported ``inference_pipelines.inference_pipeline_tgn`` from the GPU: its
    ``InferencePipeLine.get_boundary_sampled_feats`` and the module's ``KDTree`` name."""
    module.InferencePipeLine.get_boundary_sampled_feats = get_boundary_sampled_feats
    module.KDTree = neighbors.KDTree
