"""GPU parity of the pointops side (FPS, kNN, gather family) -- bit-exact for indices and
forward values -- against (a) the CPU oracle and (b) the reference's own kernels compiled
verbatim (oracle/_ref), on seeded inputs.  The reference kernels' outputs are stored in tests/golden/ref_live_pointops.npz
(oracle/golden.py: recorded by a run with TGN_GOLDEN_RECORD set where oracle/_ref is built)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import golden, oracle, ref_cuda
from toothgroupnetwork_b200 import _lib as L
from toothgroupnetwork_b200 import clouds, pointops, pointops_cuda

pytestmark = pytest.mark.gpu
G = golden.Golden("ref_live_pointops")


def assert_exact(key, got, compute):
    assert G.exact(key, got, compute), f"{key}: {G.mismatch(key, got)}"


def reference(call):
    """the reference kernel's outputs, computed once and only when they are recorded: reference(call)(i) -> output i"""
    out = []

    def get(i):
        if not out:
            out.extend(call())
        return out[i]
    return get


def dev(a, dtype=None):
    t = torch.as_tensor(a)
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


def i32(a):
    return dev(np.asarray(a, np.int32))


# ------------------------------------------------------------------------------------ FPS
FPS_CASES = [
    # (name, cloud builder, sizes, samples)
    ("cube24k_4096", lambda: [clouds.cube(24000, 0)], [4096]),          # BASELINE config C1
    ("arch24k_1024", lambda: [clouds.dental_arch(24000, 0)[0]], [1024]),
    ("dups", lambda: [clouds.with_duplicates(clouds.cube(6000, 5), 5)], [3000]),
    ("ragged", lambda: [clouds.cube(3072, 1), clouds.cube(700, 2), clouds.cube(93, 3), clouds.cube(1500, 4)], [768, 175, 23, 375]),
    ("tiny", lambda: [clouds.cube(12, 6), clouds.cube(1, 7), clouds.cube(5, 8)], [5, 1, 5]),
    ("crops16x3072", lambda: [clouds.dental_arch(3072, 10 + i)[0] for i in range(16)], [768] * 16),
    ("more_samples_than_unique", lambda: [clouds.with_duplicates(clouds.cube(40, 9), 9)], [80]),
    ("raw_mesh_100k", lambda: [clouds.dental_arch(100000, 12)[0]], [1500]),                 # SURVEY 8(f) next-2 size
    ("raw_mesh_200k", lambda: [clouds.dental_arch(200000, 15)[0]], [1200]),                # 3125 buckets: 7 per lane at 16 warps
    ("flat_and_tiny_extent", lambda: [clouds.cube(9000, 13) * torch.tensor([1.0, 1e-3, 0.0])], [700]),  # degenerate bbox
    ("arch_dups_24k", lambda: [clouds.with_duplicates(clouds.dental_arch(12000, 14)[0], 14)], [2048]),
]


def _pack(cl, ms):
    xyz = torch.cat(cl, 0).contiguous()
    offset = np.cumsum([c.shape[0] for c in cl]).astype(np.int32)
    new_offset = np.cumsum(ms).astype(np.int32)
    return xyz, offset, new_offset


@pytest.mark.parametrize("name,build,ms", FPS_CASES, ids=[c[0] for c in FPS_CASES])
@pytest.mark.parametrize("mode", [0, 1, 2, 4, 8, 201, 202, 204, 208, -1, -2, -3, -42, -44, -48, -56, -72, -84, -88, -96, -112])   # 100*G + CS; -(40 + W): single-barrier bucket schedule; -(80 + W): + register-resident tables
def test_fps_matches_oracle(name, build, ms, mode):
    cl = build()
    xyz, offset, new_offset = _pack(cl, ms)
    n_max = max(c.shape[0] for c in cl)
    want = oracle.furthestsampling(xyz.numpy(), offset, new_offset)
    try:
        got = pointops.fps_packed(xyz.cuda(), i32(offset), i32(new_offset), n_max, int(new_offset[-1]), mode)
    except L.TgnError as e:
        if mode > 0 and "no resident kernel of shape" in str(e):
            pytest.skip("cluster size not applicable to this cloud size")
        if mode <= -81 and "has no shape" in str(e):
            pytest.skip("cloud has more buckets per lane than the register-resident kernel holds")
        raise
    torch.cuda.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.mark.parametrize("name,build,ms", FPS_CASES, ids=[c[0] for c in FPS_CASES])
def test_fps_matches_reference_kernel(name, build, ms):
    cl = build()
    xyz, offset, new_offset = _pack(cl, ms)
    n_max = max(c.shape[0] for c in cl)
    x, o, no = xyz.cuda(), i32(offset), i32(new_offset)
    ref = reference(lambda: ref_cuda.furthestsampling(x, o, no, n_max, int(new_offset[-1])))
    got = pointops.furthestsampling(x, o, no)
    assert_exact(f"fps_{name}_idx", got, lambda: ref(0))
    # the oracle reproduces the reference kernel too (idx AND the final running minima, bitwise)
    o_idx, o_tmp = oracle.furthestsampling(xyz.numpy(), offset, new_offset, return_tmp=True)
    assert_exact(f"fps_{name}_idx", o_idx, lambda: ref(0))
    assert_exact(f"fps_{name}_tmp", o_tmp, lambda: ref(1))


def test_fps_drop_in_launcher_and_tmp_writeback():
    """The reference's extern "C" symbol, raw pointers, legacy stream, tmp in/out."""
    xyz = clouds.cube(5000, 11).cuda()
    o, no = i32([5000]), i32([600])
    idx = torch.zeros(600, dtype=torch.int32, device="cuda")
    tmp = torch.full((5000,), 1e10, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    lib = L.load()
    lib.furthestsampling_cuda_launcher.restype = None
    lib.furthestsampling_cuda_launcher(1, 5000, ctypes.c_void_p(xyz.data_ptr()), ctypes.c_void_p(o.data_ptr()),
                                       ctypes.c_void_p(no.data_ptr()), ctypes.c_void_p(tmp.data_ptr()), ctypes.c_void_p(idx.data_ptr()))
    torch.cuda.synchronize()
    w_idx, w_tmp = oracle.furthestsampling(xyz.cpu().numpy(), [5000], [600], return_tmp=True)
    assert np.array_equal(idx.cpu().numpy(), w_idx)
    assert np.array_equal(tmp.cpu().numpy().view(np.uint32), w_tmp.view(np.uint32))
    # pybind-style module, same buffers convention
    idx2 = torch.zeros_like(idx)
    tmp2 = torch.full_like(tmp, 1e10)
    pointops_cuda.furthestsampling_cuda(1, 5000, xyz, o, no, tmp2, idx2)
    assert torch.equal(idx2, idx) and torch.equal(tmp2, tmp)


def test_fps_full_size_properties():
    """BASELINE size (24k -> 4096) through properties that do not need the oracle: unique ids,
    first = 0, and the selected points' distance-to-set is non-increasing."""
    xyz = clouds.dental_arch(24000, 42)[0].cuda()
    idx = pointops.furthestsampling(xyz, i32([24000]), i32([4096])).long()
    assert idx[0].item() == 0 and idx.unique().numel() == 4096
    sel = xyz[idx].double()
    d = torch.cdist(sel, sel)
    gaps = torch.stack([d[i, :i].min() for i in range(1, 512)])
    assert bool((gaps[1:] <= gaps[:-1] + 1e-9).all())


# ------------------------------------------------------------------------------------ kNN
KNN_CASES = [
    ("self_k16", lambda: clouds.cube(4096, 1), None, [4096], None, 16),
    ("self_k36", lambda: clouds.dental_arch(6000, 2)[0], None, [6000], None, 36),
    ("down_k24", lambda: clouds.cube(6000, 3), 1500, [6000], [1500], 24),
    ("dups_k8", lambda: clouds.with_duplicates(clouds.cube(1500, 4), 4), None, [3000], None, 8),
    ("two_segments_k3", lambda: clouds.cube(3000, 5), 800, [1000, 3000], [300, 800], 3),
    ("short_segment_k24", lambda: clouds.cube(12 + 500, 6), None, [12, 512], None, 24),
    ("k1", lambda: clouds.cube(2000, 7), 500, [2000], [500], 1),
    ("k64", lambda: clouds.cube(1000, 8), None, [1000], None, 64),
    ("k100", lambda: clouds.cube(700, 9), None, [700], None, 100),
]


def _knn_inputs(build, m, off, noff):
    xyz = build()
    new_xyz = xyz if m is None else None
    if m is not None:
        # queries: the first points of each segment (as FPS-style subsets are drawn from the cloud)
        starts = [0] + list(off[:-1])
        q_counts = np.diff([0] + list(noff))
        new_xyz = torch.cat([xyz[s:s + c] for s, c in zip(starts, q_counts)], 0).contiguous()
    noff = off if noff is None else noff
    return xyz, new_xyz, np.asarray(off, np.int32), np.asarray(noff, np.int32)


@pytest.mark.parametrize("name,build,m,off,noff,k", KNN_CASES, ids=[c[0] for c in KNN_CASES])
def test_knn_matches_oracle(name, build, m, off, noff, k):
    xyz, new_xyz, off, noff = _knn_inputs(build, m, off, noff)
    w_idx, w_dist, w_d2 = oracle.knnquery(k, xyz.numpy(), new_xyz.numpy(), off, noff)
    idx, d2 = pointops.knn_packed(k, xyz.cuda(), new_xyz.cuda(), i32(off), i32(noff))
    assert np.array_equal(d2.cpu().numpy().view(np.uint32), w_d2.view(np.uint32))
    assert np.array_equal(idx.cpu().numpy(), w_idx)
    idx2, dist = pointops.knnquery(k, xyz.cuda(), new_xyz.cuda(), i32(off), i32(noff))
    assert torch.equal(idx2, idx)
    assert np.array_equal(dist.cpu().numpy().view(np.uint32), w_dist.view(np.uint32))


@pytest.mark.parametrize("name,build,m,off,noff,k", KNN_CASES, ids=[c[0] for c in KNN_CASES])
def test_knn_matches_reference_kernel(name, build, m, off, noff, k):
    xyz, new_xyz, off, noff = _knn_inputs(build, m, off, noff)
    x, q, o, no = xyz.cuda(), new_xyz.cuda(), i32(off), i32(noff)
    ref = reference(lambda: ref_cuda.knnquery(k, x, q, o, no))
    idx, d2 = pointops.knn_packed(k, x, q, o, no)
    assert_exact(f"knn_{name}_d2", d2, lambda: ref(1))              # float32, bit for bit
    assert_exact(f"knn_{name}_idx", idx, lambda: ref(0))
    w_idx, _, w_d2 = oracle.knnquery(k, xyz.numpy(), new_xyz.numpy(), off, noff)
    assert_exact(f"knn_{name}_idx", w_idx, lambda: ref(0))
    assert_exact(f"knn_{name}_d2", w_d2, lambda: ref(1))


GRID_CASES = [
    # name, cloud builder, offsets, query builder (None = self), new offsets, k
    ("arch24k_self_k36", lambda: clouds.dental_arch(24000, 1)[0], [24000], None, None, 36),
    ("arch24k_self_k24", lambda: clouds.dental_arch(24000, 2)[0], [24000], None, None, 24),
    ("down_6000_from_24k_k24", lambda: clouds.dental_arch(24000, 3)[0], [24000], lambda x: x[::4].contiguous(), [6000], 24),
    ("up_24k_from_6000_k3", lambda: clouds.dental_arch(24000, 4)[0][::4].contiguous(), [6000], lambda x: clouds.dental_arch(24000, 4)[0], [24000], 3),
    ("up_24k_from_6000_k1", lambda: clouds.dental_arch(24000, 5)[0][::4].contiguous(), [6000], lambda x: clouds.dental_arch(24000, 5)[0], [24000], 1),
    ("crops_16x3072_self_k36", lambda: torch.cat([clouds.dental_arch(3072, 10 + j)[0] for j in range(16)]), [3072 * (j + 1) for j in range(16)], None, None, 36),
    ("ragged_segments_k24", lambda: torch.cat([clouds.cube(n, 30 + n) for n in (12, 3000, 1, 5000, 700)]), list(np.cumsum([12, 3000, 1, 5000, 700])), None, None, 24),
    ("duplicated_vertices_k8", lambda: clouds.with_duplicates(clouds.cube(4096, 4), 4), [8192], None, None, 8),
    ("duplicated_vertices_k36", lambda: clouds.with_duplicates(clouds.dental_arch(6000, 6)[0], 5), [12000], None, None, 36),
    ("queries_outside_the_cloud_k16", lambda: clouds.cube(8000, 7) * 0.2, [8000], lambda x: clouds.cube(2000, 8) * 3.0, [2000], 16),
    ("flat_cloud_k16", lambda: clouds.cube(6000, 9) * torch.tensor([1.0, 1.0, 0.0]), [6000], None, None, 16),
    ("all_points_equal_k8", lambda: torch.ones(3000, 3), [3000], None, None, 8),
    ("k100", lambda: clouds.dental_arch(9000, 11)[0], [9000], None, None, 100),
]


@pytest.mark.parametrize("name,build,off,qbuild,noff,k", GRID_CASES, ids=[c[0] for c in GRID_CASES])
def test_knn_grid_equals_bruteforce_kernel_and_reference(name, build, off, qbuild, noff, k):
    """The uniform-grid search (csrc/knn_grid.cu) against the brute-force warp kernel (csrc/knn.cu), bit for bit --
    indices including the reference's tie order -- and against the verbatim reference kernel."""
    xyz = build().contiguous()
    q = xyz if qbuild is None else qbuild(xyz).contiguous()
    o, no = i32(np.asarray(off, np.int32)), i32(np.asarray(off if noff is None else noff, np.int32))
    x, qq = xyz.cuda(), q.cuda()
    pointops.clear_knn_caches()
    pointops.set_knn_grid(False)
    try:
        b_idx, b_d2 = pointops.knn_packed(k, x, qq, o, no)
    finally:
        pointops.set_knn_grid(True)
    launches = L.launch_count()
    g_idx, g_d2 = pointops.knn_packed(k, x, qq, o, no)
    assert L.launch_count() - launches == 5        # four build kernels + the query
    assert torch.equal(g_d2.view(torch.int32), b_d2.view(torch.int32))
    assert torch.equal(g_idx, b_idx)
    launches = L.launch_count()
    c_idx, c_d2 = pointops.knn_packed(k, x, qq, o, no)           # identical repeated query: served from the cache
    assert L.launch_count() == launches and c_idx is g_idx
    k2 = k // 2 if k > 1 else 2
    h_idx, _ = pointops.knn_packed(k2, x, qq, o, no)             # same grid, other k: one launch
    assert L.launch_count() - launches == 1
    kk = min(k, k2)
    assert torch.equal(h_idx[:, :kk], b_idx[:, :kk]) or name.startswith(("duplicated", "all_points"))
    ref = reference(lambda: ref_cuda.knnquery(k, x, qq, o, no))
    assert_exact(f"knn_grid_{name}_d2", g_d2, lambda: ref(1))
    assert_exact(f"knn_grid_{name}_idx", g_idx, lambda: ref(0))
    x.add_(0.0)                                                   # in-place write bumps the version: caches must miss
    launches = L.launch_count()
    pointops.knn_packed(k, x, qq if qbuild is not None else x, o, no)
    assert L.launch_count() - launches == 5


def test_knn_full_size_property():
    """24k x 24k, k=36: row 0 is the query itself at distance 0 and rows are sorted."""
    xyz = clouds.dental_arch(24000, 1)[0].cuda()
    o = i32([24000])
    idx, d2 = pointops.knn_packed(36, xyz, xyz, o, o)
    assert bool((d2[:, 0] == 0).all()) and bool((d2[:, 1:] >= d2[:, :-1]).all())
    assert bool((xyz[idx[:, 0].long()] == xyz).all())


# ------------------------------------------------------------------------------------ gather family
def _rand(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g)


@pytest.mark.parametrize("c", [3, 32, 35])
def test_grouping_forward_backward(c):
    n, m, k = 2000, 500, 24
    inp = _rand((n, c), 1)
    idx = torch.randint(0, n, (m, k), generator=torch.Generator().manual_seed(2), dtype=torch.int32)
    x = inp.cuda().requires_grad_(True)
    out = pointops.grouping(x, idx.cuda())
    assert np.array_equal(out.detach().cpu().numpy(), oracle.grouping_forward(inp.numpy(), idx.numpy()))
    go = _rand((m, k, c), 3)
    out.backward(go.cuda())
    want = oracle.grouping_backward(go.numpy(), idx.numpy(), n)
    np.testing.assert_allclose(x.grad.cpu().numpy(), want, rtol=1e-5, atol=1e-5)
    assert_exact(f"grouping_{c}", out, lambda: ref_cuda.grouping_forward(inp.cuda(), idx.cuda()))


def test_interpolation_kernels():
    m, n, c, k = 600, 2400, 32, 3
    inp = _rand((m, c), 1)
    idx = torch.randint(0, m, (n, k), generator=torch.Generator().manual_seed(2), dtype=torch.int32)
    w = torch.rand(n, k, generator=torch.Generator().manual_seed(3))
    out = torch.zeros(n, c, device="cuda")
    pointops_cuda.interpolation_forward_cuda(n, c, k, inp.cuda(), idx.cuda(), w.cuda(), out)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), oracle.interpolation_forward(inp.numpy(), idx.numpy(), w.numpy()).view(np.uint32))
    go = _rand((n, c), 4)
    gi = torch.zeros(m, c, device="cuda")
    pointops_cuda.interpolation_backward_cuda(n, c, k, go.cuda(), idx.cuda(), w.cuda(), gi)
    np.testing.assert_allclose(gi.cpu().numpy(), oracle.interpolation_backward(go.numpy(), idx.numpy(), w.numpy(), m), rtol=1e-4, atol=1e-5)
    assert_exact("interpolation", out, lambda: ref_cuda.interpolation_forward(inp.cuda(), idx.cuda(), w.cuda()))


@pytest.mark.parametrize("c", [32, 6])
def test_subtraction(c):
    n, k = 1500, 16
    a, b = _rand((n, c), 1), _rand((n, c), 2)
    idx = torch.randint(0, n, (n, k), generator=torch.Generator().manual_seed(3), dtype=torch.int32)
    x1, x2 = a.cuda().requires_grad_(True), b.cuda().requires_grad_(True)
    out = pointops.subtraction(x1, x2, idx.cuda())
    assert np.array_equal(out.detach().cpu().numpy(), oracle.subtraction_forward(a.numpy(), b.numpy(), idx.numpy()))
    go = _rand((n, k, c), 4)
    out.backward(go.cuda())
    g1, g2 = oracle.subtraction_backward(idx.numpy(), go.numpy())
    np.testing.assert_allclose(x1.grad.cpu().numpy(), g1, rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(x2.grad.cpu().numpy(), g2, rtol=1e-4, atol=1e-5)
    assert_exact(f"subtraction_{c}", out, lambda: ref_cuda.subtraction_forward(a.cuda(), b.cuda(), idx.cuda()))


def test_aggregation():
    n, k, c, w_c = 1200, 16, 32, 4
    inp, pos, w = _rand((n, c), 1), _rand((n, k, c), 2), _rand((n, k, w_c), 3)
    idx = torch.randint(0, n, (n, k), generator=torch.Generator().manual_seed(4), dtype=torch.int32)
    ti, tp, tw = inp.cuda().requires_grad_(True), pos.cuda().requires_grad_(True), w.cuda().requires_grad_(True)
    out = pointops.aggregation(ti, tp, tw, idx.cuda())
    assert np.array_equal(out.detach().cpu().numpy().view(np.uint32),
                          oracle.aggregation_forward(inp.numpy(), pos.numpy(), w.numpy(), idx.numpy()).view(np.uint32))
    go = _rand((n, c), 5)
    out.backward(go.cuda())
    gi, gp, gw = oracle.aggregation_backward(inp.numpy(), pos.numpy(), w.numpy(), idx.numpy(), go.numpy())
    np.testing.assert_allclose(ti.grad.cpu().numpy(), gi, rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(tp.grad.cpu().numpy(), gp, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(tw.grad.cpu().numpy(), gw, rtol=1e-4, atol=1e-4)
    assert_exact("aggregation", out, lambda: ref_cuda.aggregation_forward(inp.cuda(), pos.cuda(), w.cuda(), idx.cuda()))


def test_queryandgroup_and_interpolation_composites():
    xyz = clouds.dental_arch(3000, 3)[0]
    feat = _rand((3000, 16), 1)
    o = np.array([3000], np.int32)
    no = np.array([750], np.int32)
    fps = oracle.furthestsampling(xyz.numpy(), o, no)
    new_xyz = xyz[torch.from_numpy(fps).long()].contiguous()
    got = pointops.queryandgroup(12, xyz.cuda(), new_xyz.cuda(), feat.cuda(), None, i32(o), i32(no), use_xyz=True)
    want = oracle.queryandgroup(12, xyz.numpy(), new_xyz.numpy(), feat.numpy(), None, o, no, True)
    assert np.array_equal(got.cpu().numpy(), want)
    # interpolation: coarse (750) -> fine (3000), k=3; fp32 within 1e-5 (the reference sums
    # k separate multiply-adds, the kernel uses an fma chain)
    cf = _rand((750, 16), 2)
    f = cf.cuda().requires_grad_(True)
    up = pointops.interpolation(new_xyz.cuda(), xyz.cuda(), f, i32(no), i32(o), 3)
    w_up, w_idx, w_w = oracle.interpolation(new_xyz.numpy(), xyz.numpy(), cf.numpy(), no, o, 3)
    np.testing.assert_allclose(up.detach().cpu().numpy(), w_up, rtol=1e-5, atol=1e-6)
    up.sum().backward()
    want_g = oracle.interpolation_backward(np.ones((3000, 16), np.float32), w_idx, w_w, 750)
    np.testing.assert_allclose(f.grad.cpu().numpy(), want_g, rtol=1e-4, atol=1e-4)
    up2 = pointops.interpolation2(new_xyz.cuda(), xyz.cuda(), cf.cuda(), i32(no), i32(o), 3)
    np.testing.assert_allclose(up2.cpu().numpy(), w_up, rtol=1e-5, atol=1e-6)


def test_cpu_tensor_is_an_error():
    with pytest.raises(L.TgnError):
        pointops.furthestsampling(clouds.cube(100, 0), torch.tensor([100], dtype=torch.int32), torch.tensor([10], dtype=torch.int32))
