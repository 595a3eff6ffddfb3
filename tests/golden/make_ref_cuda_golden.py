"""Generate tests/golden/ref_cuda_*.npz by running the REFERENCE'S OWN CUDA KERNELS (compiled
verbatim for sm_100a into oracle/_ref/libpointops_ref.so by ``make -C oracle ref``) on a B200:

    gpurun -- 'python tests/golden/make_ref_cuda_golden.py gpurun_out/golden'
    cp gpurun_out/golden/ref_cuda_*.npz tests/golden/

Inputs are regenerated from seeds by the tests (toothgroupnetwork_b200.clouds), only the reference
outputs are stored.  These fixtures pin the CPU oracle (tests/test_oracle_golden.py) against the
real kernels: FPS indices + final running minima, kNN indices + squared distances (bitwise), the
gather-family forwards (bitwise).  The large kNN and gather outputs are stored as digests with a sample
(oracle/golden.pack).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import golden, ref_cuda  # noqa: E402
from toothgroupnetwork_b200 import clouds  # noqa: E402

FPS_CASES = {
    # name: (list of (generator, n, seed), samples)
    "cube24k_4096": ([("cube", 24000, 0)], [4096]),
    "arch24k_1024": ([("arch", 24000, 0)], [1024]),
    "dups6k": ([("dups", 6000, 5)], [3000]),
    "ragged": ([("cube", 3072, 1), ("cube", 700, 2), ("cube", 93, 3), ("cube", 1500, 4)], [768, 175, 23, 375]),
    "tiny": ([("cube", 12, 6), ("cube", 1, 7), ("cube", 5, 8)], [5, 1, 5]),
}
KNN_CASES = {
    # name: (generator, n, seed, offsets, query count per segment or None (=self), k)
    "self_k16": ("cube", 4096, 1, [4096], None, 16),
    "arch_k36": ("arch", 6000, 2, [6000], None, 36),
    "dups_k8": ("dups", 1500, 4, [3000], None, 8),
    "two_segments_k3": ("cube", 3000, 5, [1000, 3000], [300, 500], 3),
    "short_segment_k24": ("cube", 512, 6, [12, 512], None, 24),
}


def make_cloud(kind, n, seed):
    if kind == "cube":
        return clouds.cube(n, seed)
    if kind == "arch":
        return clouds.dental_arch(n, seed)[0]
    if kind == "dups":
        return clouds.with_duplicates(clouds.cube(n, seed), seed)
    raise ValueError(kind)


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    assert ref_cuda.available() and torch.cuda.is_available()
    fix = {}
    for name, (parts, ms) in FPS_CASES.items():
        cl = [make_cloud(*p) for p in parts]
        xyz = torch.cat(cl, 0).contiguous().cuda()
        off = torch.tensor(np.cumsum([c.shape[0] for c in cl]), dtype=torch.int32).cuda()
        noff = torch.tensor(np.cumsum(ms), dtype=torch.int32).cuda()
        idx, tmp = ref_cuda.furthestsampling(xyz, off, noff, max(c.shape[0] for c in cl), int(sum(ms)))
        fix[f"{name}_idx"] = idx.cpu().numpy()
        fix[f"{name}_tmp"] = tmp.cpu().numpy()
    np.savez_compressed(os.path.join(out_dir, "ref_cuda_fps.npz"), **fix)

    fix = {}
    for name, (kind, n, seed, offs, qcounts, k) in KNN_CASES.items():
        xyz = make_cloud(kind, n, seed)
        if qcounts is None:
            q, noffs = xyz, offs
        else:
            starts = [0] + offs[:-1]
            q = torch.cat([xyz[s:s + c] for s, c in zip(starts, qcounts)], 0).contiguous()
            noffs = list(np.cumsum(qcounts))
        idx, d2 = ref_cuda.knnquery(k, xyz.cuda(), q.cuda(), torch.tensor(offs, dtype=torch.int32).cuda(),
                                    torch.tensor(noffs, dtype=torch.int32).cuda())
        fix[f"{name}_idx"] = idx.cpu().numpy()
        fix[f"{name}_d2"] = d2.cpu().numpy()
    np.savez_compressed(os.path.join(out_dir, "ref_cuda_knn.npz"), **{e: v for k, a in fix.items() for e, v in golden.pack(k, a).items()})

    # gather family forwards on seeded random tensors
    g = torch.Generator().manual_seed(0)
    n, m, k, c, w_c = 1500, 400, 16, 32, 4
    inp = torch.randn(n, c, generator=g)
    idx = torch.randint(0, n, (m, k), generator=g, dtype=torch.int32)
    w3 = torch.rand(m, 3, generator=g)
    idx3 = torch.randint(0, n, (m, 3), generator=g, dtype=torch.int32)
    in2 = torch.randn(n, c, generator=g)
    idxn = torch.randint(0, n, (n, k), generator=g, dtype=torch.int32)
    pos = torch.randn(n, k, c, generator=g)
    wgt = torch.randn(n, k, w_c, generator=g)
    fix = {
        "grouping": ref_cuda.grouping_forward(inp.cuda(), idx.cuda()).cpu().numpy(),
        "interpolation": ref_cuda.interpolation_forward(inp.cuda(), idx3.cuda(), w3.cuda()).cpu().numpy(),
        "subtraction": ref_cuda.subtraction_forward(inp.cuda(), in2.cuda(), idxn.cuda()).cpu().numpy(),
        "aggregation": ref_cuda.aggregation_forward(inp.cuda(), pos.cuda(), wgt.cuda(), idxn.cuda()).cpu().numpy(),
    }
    np.savez_compressed(os.path.join(out_dir, "ref_cuda_gather.npz"), **{e: v for k, a in fix.items() for e, v in golden.pack(k, a).items()})
    for f in sorted(os.listdir(out_dir)):
        print(f, os.path.getsize(os.path.join(out_dir, f)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden"))
