"""The CPU oracle against fixtures produced by the reference's OWN CUDA kernels (compiled verbatim
for sm_100a, run on a B200 by tests/golden/make_ref_cuda_golden.py).  Everything bitwise."""
import importlib.util
import os

import numpy as np
import pytest
import torch

from oracle import golden, oracle

_spec = importlib.util.spec_from_file_location("make_ref_cuda_golden",
                                               os.path.join(os.path.dirname(__file__), "golden", "make_ref_cuda_golden.py"))
gen = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(gen)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


@pytest.mark.parametrize("name", sorted(gen.FPS_CASES))
def test_fps_oracle_equals_reference_kernel(golden_dir, name):
    fix = _load(golden_dir, "ref_cuda_fps.npz")
    parts, ms = gen.FPS_CASES[name]
    cl = [gen.make_cloud(*p) for p in parts]
    xyz = torch.cat(cl, 0).numpy()
    off = np.cumsum([c.shape[0] for c in cl]).astype(np.int32)
    noff = np.cumsum(ms).astype(np.int32)
    idx, tmp = oracle.furthestsampling(xyz, off, noff, return_tmp=True)
    assert np.array_equal(idx, fix[f"{name}_idx"])
    assert np.array_equal(tmp.view(np.uint32), fix[f"{name}_tmp"].view(np.uint32))


@pytest.mark.parametrize("name", sorted(gen.KNN_CASES))
def test_knn_oracle_equals_reference_kernel(golden_dir, name):
    fix = golden.Golden("ref_cuda_knn", record=False)
    kind, n, seed, offs, qcounts, k = gen.KNN_CASES[name]
    xyz = gen.make_cloud(kind, n, seed)
    if qcounts is None:
        q, noffs = xyz, offs
    else:
        starts = [0] + offs[:-1]
        q = torch.cat([xyz[s:s + c] for s, c in zip(starts, qcounts)], 0)
        noffs = list(np.cumsum(qcounts))
    idx, _, d2 = oracle.knnquery(k, xyz.numpy(), q.numpy(), np.asarray(offs, np.int32), np.asarray(noffs, np.int32))
    assert fix.exact(f"{name}_d2", d2, None), fix.mismatch(f"{name}_d2", d2)          # float32, bit for bit
    assert fix.exact(f"{name}_idx", idx, None), fix.mismatch(f"{name}_idx", idx)


def test_gather_family_oracle_equals_reference_kernels(golden_dir):
    fix = golden.Golden("ref_cuda_gather", record=False)
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
    for key, got in (("grouping", oracle.grouping_forward(inp.numpy(), idx.numpy())),
                     ("interpolation", oracle.interpolation_forward(inp.numpy(), idx3.numpy(), w3.numpy())),
                     ("subtraction", oracle.subtraction_forward(inp.numpy(), in2.numpy(), idxn.numpy())),
                     ("aggregation", oracle.aggregation_forward(inp.numpy(), pos.numpy(), wgt.numpy(), idxn.numpy()))):
        assert fix.exact(key, got, None), (key, fix.mismatch(key, got))                   # float32, bit for bit
