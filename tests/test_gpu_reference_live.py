"""GPU parity against the REFERENCE ITSELF on a B200: the reference's unmodified ``pointnet2_utils.py`` / ``pointops.py`` /
``models/modules/*.py`` on the verbatim ``pointops`` kernels of ``oracle/_ref``.  What the CPU fixtures cannot pin -- the
reference's CUDA arithmetic (cuBLAS K=3 products, the layout-dependent rounding of torch.sum(p ** 2, -1), cuDNN convolutions
with batch-statistics BatchNorm) -- is pinned here, with the call patterns the reference's modules actually use.

The reference's side of each operator- and layer-level comparison comes from ``tests/golden/ref_live_gpu.npz``, written by a
run of this file with ``TGN_GOLDEN_RECORD`` set where the reference is staged (``oracle/golden.py``); those tests need nothing
outside the repository.  The whole-model tests run the reference's model code on both operator sets and are skipped where
that code is not staged (``oracle/_ref/reference_py.tgz``, packed by ``__graft_entry__.build()`` beside a reference checkout)."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import golden, ref_cuda, ref_models
from test_gpu_blocks import Down, Layer
from toothgroupnetwork_b200 import blocks_fused, clouds
from toothgroupnetwork_b200 import pointnet2_utils as pn2

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not (ref_models.available() and ref_cuda.available()),
                                     reason="the reference's model code is not staged")
REL_TOL = 1e-4
FLOOR = 0.05      # element-wise |a-b| / max(|b|, FLOOR * max|b|)
G = golden.Golden("ref_live_gpu")

_world = {}


def world(ops):
    if ops not in _world:
        _world[ops] = ref_models.World(ops)
    return _world[ops]


def refpn():
    return world("reference").mod("external_libs.pointnet2_utils.pointnet2_utils")


def elementwise(a, b):
    """``b`` is the reference: a tensor, or a ``golden.Sampled`` (then over its sampled elements, scaled by its max |b|)."""
    if isinstance(b, golden.Sampled):
        a, scale, b = torch.from_numpy(b.pick(a)).double(), b.absmax + 1e-30, torch.from_numpy(b.values).double()
    else:
        a, b = a.detach().double(), b.detach().double()
        scale = float(b.abs().max()) + 1e-30
    a, b = a.to(b.device), b
    return float(((a - b).abs() / b.abs().clamp(min=FLOOR * scale)).max())


def assert_exact(key, got, compute):
    assert G.exact(key, got, compute), f"{key}: {G.mismatch(key, got)}"


@pytest.fixture(autouse=True)
def _fp32_library_convs():
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    pn2.set_reference_device("cuda")
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


def arch(B, N):
    return torch.stack([clouds.arch_features(N, s)[0] for s in range(B)]).cuda()      # (B,6,N)


def ref_fps_points(x1v, S):
    """The reference's farthest_point_sample + index_points on (B,N,3) arch clouds (seeds 0..B-1; one fixture per N, S)."""
    B, N = x1v.shape[0], x1v.shape[1]
    Bmax = 16 if N == 24000 else 2

    def compute():
        v = arch(Bmax, N)[:, :3, :].permute(0, 2, 1)
        with world("reference"):
            return refpn().farthest_point_sample(v, S).int()
    idx = torch.from_numpy(G.array(f"fps_{N}_{S}", compute)[:B]).long().cuda()
    return x1v[torch.arange(B, device="cuda")[:, None], idx]                              # (B,S,3), contiguous


# ------------------------------------------------------------------------------------ ball query / 3-NN: indices bit-exact
@pytest.mark.parametrize("B", [1, 16])
@pytest.mark.parametrize("r,K", [(0.025, 32), (0.05, 64), (0.1, 32), (0.2, 64)])
@pytest.mark.parametrize("pattern", ["module", "contiguous"])
def test_ball_query_bit_exact_vs_reference_on_gpu(B, r, K, pattern):
    """``module``: the layouts PointNetSetAbstraction(Msg).forward produces (xyz = permuted view of the (B,3,N) slice of
    the feature tensor, new_xyz = contiguous index_points output); ``contiguous``: both operands contiguous."""
    feats = arch(B, 24000)
    xyz = feats[:, :3, :].permute(0, 2, 1)                                  # view, strides (6N, 1, N)
    new_xyz = ref_fps_points(xyz, 1024)
    if pattern == "contiguous":
        xyz = xyz.contiguous()

    def want():
        with world("reference"):
            return refpn().query_ball_point(r, K, xyz, new_xyz)
    got = pn2.query_ball_point(r, K, xyz, new_xyz)
    assert_exact(f"ball_B{B}_r{r}_K{K}_{pattern}", got, want)


@pytest.mark.parametrize("pattern", ["views", "contiguous", "mixed"])
def test_square_distance_kernel_bitwise_vs_reference_on_gpu(pattern):
    """pointnet2_utils.square_distance (:20-41) as the losses and tsegnet.get_ddf call it: the kernel against the reference's
    matmul + two reductions on the GPU, for the layouts that change torch's |p|^2 rounding."""
    feats = arch(2, 6000)
    a = feats[:, :3, :].permute(0, 2, 1)                   # strided view (B,N,3)
    b = a[:, :512, :].contiguous()
    if pattern == "contiguous":
        a = a.contiguous()
    elif pattern == "views":
        b = b.permute(0, 2, 1).contiguous().permute(0, 2, 1)

    def want():
        with world("reference"):
            return refpn().square_distance(a, b)
    before = pn2.L.launch_count()
    got = pn2.square_distance(a, b)
    assert pn2.L.launch_count() == before + 1
    assert_exact(f"sqd_{pattern}", got, want)
    # tsegnet.get_ddf (tsegnet.py:24-33): crops (8,3072,3) as a permuted view against one centre each, (1,8,3).permute(1,0,2)
    crops = feats[:1, :3, :3072].expand(8, 3, 3072).contiguous().permute(0, 2, 1)
    centres = torch.from_numpy(G.array(f"sqd_centres_{pattern}", lambda: torch.rand(1, 8, 3))).cuda().permute(1, 0, 2)

    def want_crops():
        with world("reference"):
            return refpn().square_distance(crops, centres)
    assert_exact(f"sqd_crops_{pattern}", pn2.square_distance(crops, centres), want_crops)
    # under autograd the torch formulation is kept (the losses differentiate through it)
    ag = a.clone().requires_grad_(True)
    pn2.square_distance(ag, b).sum().backward()
    assert ag.grad is not None


@pytest.mark.parametrize("pattern", ["views", "contiguous", "mixed"])
def test_three_nn_bit_exact_vs_reference_on_gpu(pattern):
    feats = arch(2, 24000)
    x1 = feats[:, :3, :].permute(0, 2, 1)
    x2 = ref_fps_points(x1, 1024)                                                     # contiguous (B,1024,3)
    if pattern == "contiguous":
        x1 = x1.contiguous()
    elif pattern == "views":
        x2 = x2.permute(0, 2, 1).contiguous().permute(0, 2, 1)                        # strided view

    def want(i):
        def compute():
            with world("reference"):
                wd, wi = refpn().square_distance(x1, x2).sort(dim=-1)
            return (wd[:, :, :3], wi[:, :, :3])[i]
        return compute
    gd, gi = pn2.three_nn(x1, x2)
    assert_exact(f"three_nn_d_{pattern}", gd, want(0))
    if not G.exact(f"three_nn_i_{pattern}", gi.long(), want(1)):                      # equal distances may swap
        assert_exact(f"three_nn_d_{pattern}", torch.gather(pn2.square_distance(x1, x2), 2, gi.long()), want(0))


def test_three_interpolate_bit_exact_vs_reference_lines_on_gpu():
    """pointnet2_utils.py:333-340 evaluated by torch on the GPU (sort, reciprocal, normalise, weighted sum) against the
    3-NN + interpolation kernels: identical bits, including the normaliser's CUDA reduce order."""
    feats = arch(2, 24000)
    x1 = feats[:, :3, :].permute(0, 2, 1)
    g = torch.Generator(device="cuda").manual_seed(9)
    x2 = ref_fps_points(x1, 1024)
    p2 = torch.randn(2, 1024, 64, device="cuda", generator=g)
    ref = {}

    def reference():
        if not ref:
            with world("reference"):
                dists = refpn().square_distance(x1, x2)
                dists, idx = dists.sort(dim=-1)
                dists, idx = dists[:, :, :3], idx[:, :, :3]
                dist_recip = 1.0 / (dists + 1e-8)
                norm = torch.sum(dist_recip, dim=2, keepdim=True)
                weight = dist_recip / norm
                ref.update(dists=dists, out=torch.sum(refpn().index_points(p2, idx) * weight.view(2, 24000, 3, 1), dim=2))
        return ref
    gd, gi = pn2.three_nn(x1, x2)
    got = pn2.three_interpolate(p2, gd, gi)
    assert_exact("interp_dists", gd, lambda: reference()["dists"])
    assert_exact("interp_out", got, lambda: reference()["out"])


# ------------------------------------------------------------------------------------ modules with batch-statistics BatchNorm
def _state(module):
    return {k: v.clone() for k, v in module.state_dict().items()}


def _copy(state, dst):
    dst.load_state_dict(state)
    return dst


@pytest.mark.parametrize("train_bn", [True, False])
@pytest.mark.parametrize("B", [1, 3])
def test_set_abstraction_ssg_vs_reference_module(train_bn, B):
    feats = arch(B, 8192)
    xyz = feats[:, :3, :]
    torch.manual_seed(0)
    ours = pn2.PointNetSetAbstraction(512, 0.1, 32, 9, [32, 32, 64], False).cuda().train(train_bn)
    state = _state(ours)
    ref = {}

    def reference():
        if not ref:
            with world("reference"), torch.no_grad():
                mod = _copy(state, refpn().PointNetSetAbstraction(512, 0.1, 32, 9, [32, 32, 64], False).cuda()).train(train_bn)
                ref["xyz"], ref["out"] = mod(xyz, feats)
                ref["bns"] = mod.mlp_bns
        return ref
    key = f"ssg_B{B}_{'train' if train_bn else 'eval'}"
    before = pn2.L.launch_count()
    with torch.no_grad():
        got_xyz, got = ours(xyz, feats)
    assert pn2.L.launch_count() > before
    assert_exact(key + "_xyz", got_xyz, lambda: reference()["xyz"])
    assert elementwise(got, G.sampled(key + "_out", lambda: reference()["out"])) < REL_TOL
    if train_bn:      # torch's side effects of a training-mode BatchNorm
        for i, a in enumerate(ours.mlp_bns):
            mean = G.array(f"{key}_bn{i}_running_mean", lambda: reference()["bns"][i].running_mean)
            var = G.array(f"{key}_bn{i}_running_var", lambda: reference()["bns"][i].running_var)
            assert elementwise(a.running_mean, torch.from_numpy(mean).cuda()) < 1e-4
            assert elementwise(a.running_var, torch.from_numpy(var).cuda()) < 1e-4
            assert int(a.num_batches_tracked) == int(G.array(f"{key}_bn{i}_batches", lambda: reference()["bns"][i].num_batches_tracked).item())


@pytest.mark.parametrize("train_bn", [True, False])
@pytest.mark.parametrize("cfg", [
    (1024, [0.025, 0.05], [32, 64], 6, [[128, 128], [128, 128]]),           # pointnet_pp.py:13 (scale 4)
    (1024, [0.025, 0.05], [32, 64], 6, [[32, 32], [32, 32]]),               # tsg_centroid_module.py:10
    (256, [0.1, 0.2], [32, 64], 6, [[196, 256], [196, 256]]),               # widths of tsg sa3 on raw features
])
def test_set_abstraction_msg_vs_reference_module(train_bn, cfg):
    feats = arch(1, 24000)
    xyz = feats[:, :3, :]
    torch.manual_seed(0)
    ours = pn2.PointNetSetAbstractionMsg(*cfg).cuda().train(train_bn)
    state = _state(ours)
    ref = {}

    def reference():
        if not ref:
            with world("reference"), torch.no_grad():
                mod = _copy(state, refpn().PointNetSetAbstractionMsg(*cfg).cuda()).train(train_bn)
                ref["xyz"], ref["out"] = mod(xyz, feats)
        return ref
    key = f"msg_{cfg[0]}_{cfg[4][0][0]}_{'train' if train_bn else 'eval'}"
    with torch.no_grad():
        got_xyz, got = ours(xyz, feats)
    assert_exact(key + "_xyz", got_xyz, lambda: reference()["xyz"])
    want_stride = G.array(key + "_xyz_stride", lambda: np.asarray(reference()["xyz"].stride(), np.int64))
    assert got_xyz.stride() == tuple(int(s) for s in want_stride)         # same view layout as the reference hands on
    assert elementwise(got, G.sampled(key + "_out", lambda: reference()["out"])) < REL_TOL


@pytest.mark.parametrize("train_bn", [True, False])
def test_group_all_wide_vs_reference_module(train_bn):
    """tsg_seg_module.py:26 flatten_sa: PointNetSetAbstraction(None, None, None, 512+3, [256, 512], True) on 256 points."""
    g = torch.Generator(device="cuda").manual_seed(3)
    xyz = torch.rand(2, 3, 256, device="cuda", generator=g)
    pts = torch.randn(2, 512, 256, device="cuda", generator=g)
    torch.manual_seed(0)
    ours = pn2.PointNetSetAbstraction(None, None, None, 515, [256, 512], True).cuda().train(train_bn)
    state = _state(ours)

    def want():
        with world("reference"), torch.no_grad():
            ref = _copy(state, refpn().PointNetSetAbstraction(None, None, None, 515, [256, 512], True).cuda()).train(train_bn)
            return ref(xyz, pts)[1]
    with torch.no_grad():
        _, got = ours(xyz, pts)
    assert elementwise(got, G.sampled(f"group_all_{'train' if train_bn else 'eval'}", want)) < REL_TOL


@pytest.mark.parametrize("train_bn", [True, False])
@pytest.mark.parametrize("shape", [(24000, 1024, 6, 128, [64, 32]), (512, 256, 512, 1024, [1024, 1024]), (1024, 1, 64, 128, [64])])
def test_feature_propagation_vs_reference_module(train_bn, shape):
    """Against the reference module on the GPU and against the same module evaluated in float64 (the exact answer):
    within 1e-4 of the reference, or -- batch-statistics BatchNorm over few rows amplifies fp32 rounding, and the
    reference's own fp32 run then sits further than 1e-4 from the exact result -- as close to the exact result as the
    reference is (factor 2)."""
    N, S, D1, D2, mlp = shape
    B = 2
    feats = arch(B, N)
    xyz1 = feats[:, :3, :]
    g = torch.Generator(device="cuda").manual_seed(5)
    x1v = xyz1.permute(0, 2, 1)
    new = ref_fps_points(x1v, S) if S >= 3 else x1v[:, :1, :].contiguous()
    xyz2 = new.permute(0, 2, 1)                                                 # the view a set-abstraction level returns
    p1 = torch.randn(B, D1, N, device="cuda", generator=g)
    p2 = torch.randn(B, D2, S, device="cuda", generator=g)
    torch.manual_seed(0)
    ours = pn2.PointNetFeaturePropagation(D1 + D2, mlp).cuda().train(train_bn)
    state = _state(ours)
    ref = {}

    def reference():
        if not ref:
            with world("reference"), torch.no_grad():
                mod = _copy(state, refpn().PointNetFeaturePropagation(D1 + D2, mlp).cuda()).train(train_bn)
                ref["want"] = mod(xyz1, xyz2, p1, p2)
                mod.load_state_dict(state)
                ref["truth"] = mod.double()(xyz1.double(), xyz2.double(), p1.double(), p2.double())
                ref["err_ref_truth"] = elementwise(ref["want"], ref["truth"])
        return ref
    key = f"fp_{N}_{S}_{'train' if train_bn else 'eval'}"
    with torch.no_grad():
        got = ours(xyz1, xyz2, p1, p2)
    want = G.sampled(key + "_out", lambda: reference()["want"])
    truth = G.sampled(key + "_truth", lambda: reference()["truth"])
    err_ref_t = float(G.array(key + "_err_ref_truth", lambda: np.float64(reference()["err_ref_truth"])).item())
    err, err_ours_t = elementwise(got, want), elementwise(got, truth)
    assert err < REL_TOL or err_ours_t <= max(REL_TOL, 2.0 * err_ref_t), (err, err_ours_t, err_ref_t)


def test_feature_propagation_forward_backward_under_autograd_bitwise():
    """Training step through PointNetFeaturePropagation (autograd on): 3-NN, interpolation (CUDA gather with the order-exact
    backward) and the reference's own conv/BN torch code -> output and every gradient bit-identical to the reference module."""
    N, S, D1, D2, mlp = 6000, 512, 6, 64, [32, 16]
    feats = arch(2, N)
    xyz1 = feats[:, :3, :]
    g = torch.Generator(device="cuda").manual_seed(7)
    xyz2 = ref_fps_points(xyz1.permute(0, 2, 1), S).permute(0, 2, 1)
    p1 = torch.randn(2, D1, N, device="cuda", generator=g)
    p2 = torch.randn(2, D2, S, device="cuda", generator=g)
    torch.manual_seed(0)
    ours = pn2.PointNetFeaturePropagation(D1 + D2, mlp).cuda().train()
    state = _state(ours)

    def step(mod):
        a1, a2 = p1.clone().requires_grad_(True), p2.clone().requires_grad_(True)
        out = mod(xyz1, xyz2, a1, a2)
        out.square().mean().backward()
        return {"out": out.detach(), "g_p1": a1.grad, "g_p2": a2.grad, **{n: q.grad for n, q in mod.named_parameters()}}
    ref = {}

    def reference():
        if not ref:
            with world("reference"):
                mod = refpn().PointNetFeaturePropagation(D1 + D2, mlp).cuda().train()
                mod.load_state_dict(state)
                ref.update(step(mod))
        return ref
    got = step(ours)
    for k in got:
        if k in ("out", "g_p1", "g_p2"):
            assert_exact("fp_grad_" + k, got[k], lambda: reference()[k])
        else:       # cuDNN's weight-gradient kernels are not bit-reproducible run to run; the inputs to them are identical
            assert elementwise(got[k], G.sampled("fp_grad_" + k, lambda: reference()[k])) < 1e-5, k


# ------------------------------------------------------------------------------------ the fused kernels behind the reference's blocks.py
def _flat_state(state):
    return torch.cat([state[k].detach().double().reshape(-1).cpu() for k in sorted(state)])


@pytest.mark.parametrize("c,K,n", [(32, 36, 24000), (64, 24, 6000), (128, 24, 1500), (512, 24, 93)])
@pytest.mark.parametrize("train_bn", [True, False])
def test_fused_point_transformer_layer_vs_reference_layer(c, K, n, train_bn):
    """blocks.PointTransformerLayer (:14-44) under no_grad: the fused multi-pass kernel (csrc/pt_layer.cu) against the reference's own
    layer on the reference's operators, and against that layer evaluated in float64 with the same neighbour indices.  Both layers
    take the same weights: the same seeded construction, checked against the reference's state."""
    name = "models.modules.cbl_point_transformer.blocks"
    p = clouds.dental_arch(n, 4)[0].cuda()
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(n, c, device="cuda", generator=g)
    o = torch.tensor([n], dtype=torch.int32, device="cuda")

    def seeded(layer):
        g2 = torch.Generator().manual_seed(3)
        with torch.no_grad():
            for b in (layer.linear_p[1], layer.linear_w[0], layer.linear_w[3]):      # non-trivial affine / running statistics
                b.weight.copy_(torch.rand(b.weight.shape, generator=g2) + 0.5)
                b.bias.copy_(torch.randn(b.bias.shape, generator=g2) * 0.1)
                b.running_mean.copy_(torch.randn(b.running_mean.shape, generator=g2) * 0.1)
                b.running_var.copy_(torch.rand(b.running_var.shape, generator=g2) + 0.5)
        return layer
    torch.manual_seed(0)
    ours = seeded(Layer(c, K)).cuda().train(train_bn)
    state = _state(ours)
    ref = {}

    def reference():
        if not ref:
            with world("reference"), torch.no_grad():
                torch.manual_seed(0)
                mod = seeded(world("reference").mod(name).PointTransformerLayer(c, c, 8, K)).cuda().train(train_bn)
                ref["state"] = _state(mod)
                ref["want"] = mod([p, x, o])
                ref["after"] = _state(mod)
                # float64 truth: same layer, same neighbour indices (kNN on the float32 coordinates)
                mod.load_state_dict(ref["state"])
                po = world("reference").mod("external_libs.pointops.functions.pointops")
                saved = po.knnquery
                po.knnquery = lambda k, xyz, new_xyz, off, noff: saved(k, xyz.float().contiguous(), new_xyz.float().contiguous(), off, noff)
                try:
                    ref["truth"] = mod.double()([p.double(), x.double(), o])
                finally:
                    po.knnquery = saved
                ref["err_ref_truth"] = elementwise(ref["want"], ref["truth"])
        return ref
    key = f"ptl_{c}_{K}_{n}_{'train' if train_bn else 'eval'}"
    assert_exact(key + "_state", _flat_state(state), lambda: _flat_state(reference()["state"]))
    with torch.no_grad():
        assert blocks_fused.pt_layer_fusable(ours, p, x, o)
        launches = pn2.L.launch_count()
        got = blocks_fused.pt_layer_forward(ours, [p, x, o])
        assert pn2.L.launch_count() - launches >= 2
    want = G.sampled(key + "_out", lambda: reference()["want"])
    truth = G.sampled(key + "_truth", lambda: reference()["truth"])
    e_ref = float(G.array(key + "_err_ref_truth", lambda: np.float64(reference()["err_ref_truth"])).item())
    err, e_ours = elementwise(got, want), elementwise(got, truth)
    assert err < REL_TOL or e_ours <= max(REL_TOL, 2.0 * e_ref), (err, e_ours, e_ref)
    if train_bn:
        for k, v in ours.state_dict().items():
            if "running" in k:
                assert elementwise(v, torch.from_numpy(G.array(f"{key}_after_{k}", lambda: reference()["after"][k])).cuda()) < 1e-4, k
            if "num_batches_tracked" in k:
                assert int(v) == int(G.array(f"{key}_after_{k}", lambda: reference()["after"][k]).item()), k


@pytest.mark.parametrize("train_bn", [True, False])
def test_fused_transition_down_vs_reference(train_bn):
    """blocks.TransitionDown (stride 4, :59-79) under no_grad on the tcgen05 layer chain: same sampled points, features within 1e-4 /
    the float64 criterion.  Both modules take the same weights: the same seeded construction, checked against the reference's state."""
    name = "models.modules.cbl_point_transformer.blocks"
    p = torch.cat([clouds.dental_arch(6000, 5)[0], clouds.dental_arch(3000, 6)[0]]).cuda()
    g = torch.Generator(device="cuda").manual_seed(4)
    x = torch.randn(9000, 32, device="cuda", generator=g)
    o = torch.tensor([6000, 9000], dtype=torch.int32, device="cuda")
    torch.manual_seed(0)
    ours = Down(32, 64, 4, 24).cuda().train(train_bn)
    ref = {}

    def reference():
        if not ref:
            with world("reference"), torch.no_grad():
                torch.manual_seed(0)
                mod = world("reference").mod(name).TransitionDown(32, 64, 4, 24).cuda().train(train_bn)
                ref["state"] = _state(mod)
                ref["p"], ref["x"], ref["o"] = mod([p, x, o])
        return ref
    key = f"td_{'train' if train_bn else 'eval'}"
    assert_exact(key + "_state", _flat_state(_state(ours)), lambda: _flat_state(reference()["state"]))
    with torch.no_grad():
        assert blocks_fused.transition_down_fusable(ours, p, x, o)
        p_new, x_new, o_new = blocks_fused.transition_down_forward(ours, [p, x, o])
    assert_exact(key + "_p", p_new, lambda: reference()["p"])
    assert_exact(key + "_o", o_new, lambda: reference()["o"])
    assert elementwise(x_new, G.sampled(key + "_x", lambda: reference()["x"])) < REL_TOL


def test_farthest_point_sample_np_wrapper():
    """pointnet2_utils.farthest_point_sample_np (:103-118; unused by the reference, random start there): numpy in/out,
    deterministic start, same samples as the tensor API."""
    xyz = clouds.dental_arch(6000, 3)[0]
    got = pn2.farthest_point_sample_np(xyz.numpy()[None], 256)
    want = pn2.farthest_point_sample(xyz[None].cuda(), 256).cpu().numpy()
    assert got.dtype == np.int64 and np.array_equal(got, want)


# ------------------------------------------------------------------------------------ the reference's own blocks.py on both operator sets
@needs_reference
def test_real_blocks_transition_down_transformer_layer_transition_up():
    """``models/modules/cbl_point_transformer/blocks.py`` as shipped (TransitionDown :47-79, PointTransformerLayer :14-44,
    TransitionUp :82-111), imported once per operator set; same weights, training-mode BatchNorm, forward + backward."""
    name = "models.modules.cbl_point_transformer.blocks"
    xyz, _, _ = clouds.dental_arch(24000, 2)
    p = xyz.cuda()
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(24000, 32, device="cuda", generator=g)
    o = torch.tensor([24000], dtype=torch.int32, device="cuda")
    outs, grads, state = {}, {}, None
    for ops in ("reference", "b200"):
        w = world(ops)
        with w:
            B = w.mod(name)
            torch.manual_seed(0)
            mods = torch.nn.ModuleDict({"td": B.TransitionDown(32, 64, 4, 24), "pt": B.PointTransformerLayer(64, 64, 8, 24),
                                        "tu": B.TransitionUp(64, 32), "lin": torch.nn.Linear(32, 32)}).cuda()
            if state is None:
                state = {k: v.clone() for k, v in mods.state_dict().items()}
            else:
                mods.load_state_dict(state)
            xin = x.clone().requires_grad_(True)
            p2, x2, o2 = mods["td"]([p, xin, o])
            x3 = mods["pt"]([p2, x2, o2])
            up = mods["tu"]([p, mods["lin"](xin), o], [p2, x3, o2])
            up.square().mean().backward()
            outs[ops] = {"p2": p2, "x2": x2, "o2": o2, "x3": x3, "up": up}
            grads[ops] = {"x": xin.grad.clone(), **{n: q.grad.clone() for n, q in mods.named_parameters() if q.grad is not None}}
    a, b = outs["b200"], outs["reference"]
    assert torch.equal(a["p2"], b["p2"]) and torch.equal(a["o2"], b["o2"])          # FPS indices identical
    for k in ("x2", "x3", "up"):
        assert elementwise(a[k], b[k]) < REL_TOL, k
    # backward: the gathers' scatter-adds follow torch's index_put order (csrc/csr.cu), everything else is the reference's
    # own torch code on bit-identical inputs -> every gradient bit-identical
    for k in ("x2", "x3", "up"):
        assert torch.equal(a[k], b[k]), k
    for k, want in grads["reference"].items():
        got = grads["b200"][k]
        assert torch.equal(got, want), (k, float((got - want).abs().max()), float(want.abs().max()))


# ------------------------------------------------------------------------------------ whole models (C2-model, C3, C4)
def _model_parity():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import model_parity
    return model_parity


@needs_reference
def test_pointnet_pp_model_eval_bn_logits_vs_reference():
    mp = _model_parity()
    feats, _ = mp.make_inputs(24000)
    res = mp.case_pp([world("reference"), world("b200")], feats, False, mp.Timer())
    assert res["indices_identical"]
    assert res["verdict"]["pass"], res["verdict"]


@needs_reference
def test_pointnet_pp_model_train_bn_logits_vs_reference():
    mp = _model_parity()
    feats, _ = mp.make_inputs(24000)
    res = mp.case_pp([world("reference"), world("b200")], feats, True, mp.Timer())
    assert res["indices_identical"]
    assert res["verdict"]["pass"], res["verdict"]


@needs_reference
def test_tgnet_fps_forward_backward_vs_reference():
    mp = _model_parity()
    feats, labels = mp.make_inputs(24000)
    res = mp.case_tgn([world("reference"), world("b200")], feats, labels, mp.Timer())
    assert res["indices_identical"]
    assert res["tensors"]["nn_crop_indexes"]["bitwise"]
    assert res["verdict"]["pass"], res["verdict"]
    assert res["grads"]["pass"], res["grads"]


@needs_reference
def test_tgnet_inference_branch_clusters_and_crops_like_the_reference():
    """The label-free branch of GroupingNetworkModule.forward (grouping_network_module.py:58-73): predicted offsets are clustered
    (ops_utils.get_clustering_labels: DBSCAN + noise vote), the centroids pick the 3072-point crops, the second network runs on them.
    Random weights predict no clusters, so the first network is replaced in BOTH worlds by the same stand-in that 'predicts' the
    foreground mask and offsets of a nearly converged model; everything after it is the reference's code on either operator set:
    scikit-learn + KDTree on the host in one world, csrc/dbscan.cu + csrc/crop_knn.cu in the other."""
    import numpy as np
    mp = _model_parity()
    n = 24000
    xyz, normal, label = clouds.dental_arch(n, 2)
    lab = torch.where(label < 0, torch.zeros_like(label), label).long()
    cent = torch.stack([xyz[lab == c].mean(0) if bool((lab == c).any()) else torch.zeros(3) for c in range(int(lab.max()) + 1)])
    g = torch.Generator().manual_seed(3)
    offset = 0.93 * (cent[lab] - xyz) + 0.003 * torch.randn(n, 3, generator=g)
    stray = torch.rand(n, generator=g) < 0.03
    offset[stray] += 0.08 * torch.randn(int(stray.sum()), 3, generator=g)
    offset[lab == 0] = 0
    sem = torch.stack([(lab == 0).float(), (lab != 0).float()]).unsqueeze(0).cuda()          # (1, 2, n) "logits"
    offset = offset.t().contiguous().unsqueeze(0).cuda()                                     # (1, 3, n)
    feats = torch.cat([xyz, normal], 1).t().contiguous().unsqueeze(0).cuda()

    class Converged(torch.nn.Module):
        def forward(self, inputs):
            return sem, offset, None, None

    outs, state = {}, None
    for w in (world("reference"), world("b200")):
        with w, torch.no_grad():
            torch.manual_seed(0)
            module = w.mod("models.modules.grouping_network_module").GroupingNetworkModule({"model_parameter": dict(mp.TGN_PARAMS)}).cuda()
            if state is None:
                state = {k: v.clone() for k, v in module.state_dict().items()}
            module.load_state_dict(state)
            module.eval()
            module.first_ins_cent_model = Converged()
            if w.ops == "b200":
                assert w.mod("ops_utils").get_clustering_labels.__module__ == "toothgroupnetwork_b200.clustering"
            outs[w.ops] = module([feats])
    ref, new = outs["reference"], outs["b200"]
    assert len(ref["nn_crop_indexes"]) == len(new["nn_crop_indexes"]) == 1
    assert np.array_equal(np.asarray(ref["nn_crop_indexes"][0]), np.asarray(new["nn_crop_indexes"][0]))
    assert np.asarray(ref["nn_crop_indexes"][0]).shape[0] >= 10                               # the teeth were found
    assert torch.equal(ref["cropped_feature_ls"], new["cropped_feature_ls"])
    assert elementwise(new["sem_2"], ref["sem_2"]) < REL_TOL            # (the second network of tgnet_fps has no offset head)
