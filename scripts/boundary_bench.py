"""Boundary stage of the tgnet inference pipeline: the reference's host method beside the device method.

At 100 000 and 200 000 raw vertices of a seeded dental arch (24 000 labelled sampled points) this times
* ``host``: the reference method (inference_pipeline_tgn.py:289-330) restated with scikit-learn's KDTree and
  gen_utils.count_unique_by_row on the host, FPS from this package, so only the host part differs;
* ``device``: ``toothgroupnetwork_b200.boundary.boundary_sampled_feats``, numpy in and numpy out;
* ``kernel``: the k = 40 kNN + label vote alone (grid built once), CUDA events;
* ``transfer_k1``: the final label transfer of :137-138 (KDTree over 44 000 labelled points, k = 1 for every raw vertex),
  scikit-learn and ``neighbors.KDTree``, tree build included in both,
and checks in the same run that both sides return the same arrays (bitwise, same numpy seed) and the same indices.
Writes one JSON with the card name, its power limit and the host CPU count read in the same run.

    python scripts/boundary_bench.py --out profiles/r3_boundary_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import boundary_oracle as B  # noqa: E402
from toothgroupnetwork_b200 import boundary, clouds, neighbors, pointops  # noqa: E402

INFO = B.BOUNDARY_INFO


def host_method(point_labels, org_feats, sampled_feats):
    from sklearn.neighbors import KDTree
    tree = KDTree(sampled_feats[:, :3].copy(), leaf_size=40)
    near = tree.query(org_feats[:, :3], k=40, return_distance=False)
    bd = B.count_unique_by_row(point_labels[near])[:, 0] / 40. < INFO["bdl_ratio"]
    k1 = tree.query(org_feats[:, :3], k=1, return_distance=False)
    ps = point_labels[k1[:, 0]].reshape(-1, 1)
    perm = np.random.permutation(int(bd.sum()))
    bd_feat, bd_lab = org_feats[bd][perm[:INFO["num_of_bdl_points"]]], ps[bd][perm[:INFO["num_of_bdl_points"]]]
    npoint = INFO["num_of_all_points"] - bd_feat.shape[0]
    non = org_feats[~bd]
    xyz = torch.from_numpy(np.array(non[:, :3])).float().cuda()                 # gen_utils.fps :135-140
    idx = pointops.furthestsampling(xyz, torch.tensor([xyz.shape[0]]).cuda().int(), torch.tensor([npoint]).cuda().int())
    f = idx.cpu().numpy().reshape(-1)
    return (np.concatenate([bd_feat, non[f]], 0), np.concatenate([bd_lab, ps[~bd][f]], 0), bd_feat, bd_lab)


def case(n: int, seed: int):
    xyz, normal, label = clouds.dental_arch(n, seed)
    org = torch.cat([xyz, normal], 1).double().numpy()
    sel = torch.randperm(n, generator=torch.Generator().manual_seed(seed + 100))[:24000].numpy()
    return (label[torch.from_numpy(sel)] + 1).double().numpy(), org, org[sel].copy(), sel


def wall(fn, reps: int):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), ts, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_boundary_bench.json"))
    ap.add_argument("--sizes", default="100000,200000")
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("boundary_bench.py needs a CUDA device")
    from sklearn.neighbors import KDTree
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi, "host_cpu_count": os.cpu_count(),
           "torch": torch.__version__, "units": "ms, median of the listed repetitions", "cases": []}
    for n in [int(s) for s in a.sizes.split(",")]:
        labels, org, sampled, sel = case(n, 50 + n // 100000)
        row = {"raw_vertices": n, "sampled_points": 24000}
        # host method vs device method, the same numpy seed, outputs compared bitwise
        np.random.seed(1)
        host_ms, host_all, want = wall(lambda: host_method(labels, org, sampled), a.host_reps)
        host_post = np.random.random()
        np.random.seed(1)
        for _ in range(2):
            boundary.boundary_sampled_feats(labels, org, sampled, **INFO)            # warm-up (module load, allocator)
        np.random.seed(1)
        dev_ms, dev_all, got = wall(lambda: boundary.boundary_sampled_feats(labels, org, sampled, **INFO), a.host_reps)
        dev_post = np.random.random()
        row["outputs_equal"] = bool(all(g.dtype == w.dtype and g.shape == w.shape and g.tobytes() == w.tobytes()
                                        for g, w in zip(got, want)))
        row["rng_state_equal"] = bool(host_post == dev_post)
        row["n_boundary_taken"] = int(want[2].shape[0])
        dev_ms, dev_all, _ = wall(lambda: boundary.boundary_sampled_feats(labels, org, sampled, **INFO), a.reps)
        row.update(host_method_ms=host_ms, host_method_all=host_all, device_method_ms=dev_ms, device_method_all=dev_all)
        # the k = 40 kernel alone
        grid = neighbors.Grid(torch.from_numpy(sampled[:, :3].copy()).cuda())
        q = torch.from_numpy(org[:, :3].copy()).cuda()
        lab = torch.from_numpy(labels).cuda()
        for _ in range(3):
            grid.label_vote(q, lab, 40, INFO["bdl_ratio"])
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        ev[0].record()
        for _ in range(a.reps):
            grid.label_vote(q, lab, 40, INFO["bdl_ratio"])
        ev[1].record()
        torch.cuda.synchronize()
        row["kernel_k40_label_vote_ms"] = ev[0].elapsed_time(ev[1]) / a.reps
        # final transfer of :137-138: 44 000 labelled points -> every raw vertex, k = 1.  The 20 000 extra rows are drawn from
        # the vertices that were not sampled, so no point is in the tree twice (a duplicate makes an exact tie, where the
        # tree's choice depends on its traversal and this package's is the lower index); rows that still differ are counted
        # and checked to be exact ties
        rest = np.setdiff1d(np.arange(n), sel)
        extra = rest[torch.randperm(rest.shape[0], generator=torch.Generator().manual_seed(n))[:20000].numpy()]
        final_pts = np.concatenate([sampled[:, :3], org[extra, :3]])
        h1_ms, h1_all, w1 = wall(lambda: KDTree(final_pts, leaf_size=2).query(org[:, :3], k=1, return_distance=False), a.host_reps)
        neighbors.KDTree(final_pts, leaf_size=2).query(org[:, :3], k=1, return_distance=False)
        d1_ms, d1_all, g1 = wall(lambda: neighbors.KDTree(final_pts, leaf_size=2).query(org[:, :3], k=1, return_distance=False), a.reps)
        diff = np.nonzero(w1[:, 0] != g1[:, 0])[0]
        def rdist_rows(i):
            d = final_pts[i] - org[diff, :3]
            return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        ties = bool(np.array_equal(rdist_rows(w1[diff, 0]), rdist_rows(g1[diff, 0])) and np.all(g1[diff, 0] < w1[diff, 0]))
        row.update(transfer_k1_host_ms=h1_ms, transfer_k1_host_all=h1_all, transfer_k1_device_ms=d1_ms, transfer_k1_device_all=d1_all,
                   transfer_k1_indices_equal=bool(diff.size == 0), transfer_k1_rows_differing=int(diff.size),
                   transfer_k1_differences_are_ties=ties)
        res["cases"].append(row)
        print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "cases"}))


if __name__ == "__main__":
    main()
