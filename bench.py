#!/usr/bin/env python
"""bench.py -- sampled-points/sec of FPS + ball query + grouped shared-MLP on 24k-point clouds.

Workload (BASELINE.json configs[1], SURVEY.md 8d "C2(i)"): PointNet++ set-abstraction level 1,
``PointNetSetAbstraction(npoint=1024, radius=0.1, nsample=32, in_channel=6+3, mlp=[32,32,64])``,
eval-mode BatchNorm, forward only, on a batch of synthetic dental-arch clouds of 24 000 points
(xyz + normals).  One step = one pass over one batch of ``--clouds`` clouds per GPU:
    FPS 24000->1024  ->  ball query (r=0.1, K=32)  ->  fused gather+MLP(9->32->32->64)+max.
metric = sampled points per second = clouds * 1024 / time, whole job (all ranks).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--clouds B] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

* ``value``: the PUBLIC module call ``sa(xyz, feats)`` with inputs resident in HBM, CUDA-event timed, max over ranks.
  ``stage_ms`` comes from a separate staged pass of the same kernels with events between the stages.
* ``e2e``: the same step through ``HostPipeline(sa)`` with HOST (pinned) inputs: H2D copy of the (B,6,N) feature
  tensor and D2H copy of both outputs inside the timed region.  Each rank binds itself and its pinned buffers to
  its GPU's NUMA node first (``numa``).
* ``roofline``: the dominant kernel (FPS), real DRAM traffic / time against the measured HBM copy peak;
  ``roofline_stages``: one entry per stage (FPS: HBM; ball query: fp32 issue; group-MLP: tensor pipe).
* ``parity_ok``: cloud 0 of this rank against the CPU oracle (indices bitwise, features element-wise 1e-4).
* ``ref_gpu``: the REFERENCE's own GPU path for the same step (verbatim FPS kernel from ``oracle/_ref`` + the reference's
  torch ball query / gather / Conv2d+BN+ReLU / max), timed with CUDA events on this GPU (rank 0, bounded batch).
* ``latency_ms``: FPS latency at B in {1,16,148,1184} x M in {1024,4096} (``c1`` = BASELINE configs[0], 24000->4096 on
  one cloud, bit-exact against the reference kernel), ``knn``: the tgnet_fps kNN launch mix beside the reference kernel.
* ``cpu_baseline`` / ``--impl reference``: the oracle's port of the reference's CPU-capable formulation of the same
  path (FPS loop + query_ball_point + grouped MLP, one cloud per host thread), bounded sample.
Inputs are larger than L2 (B*24000*6*4 bytes = 682 MB at the default B = 1184); no explicit flush.
* ``--dump-outputs DIR``: after the timed steps, rank 0 writes what the last timed ``sa(xyz, feats)`` returned, for the same
  seeded sample of at most ``DUMP_CLOUDS`` clouds every run, as float32 ``DIR/new_xyz.npy`` (n, 3, 1024) and
  ``DIR/new_points.npy`` (n, 64, 1024), with the cloud indices in ``DIR/cloud_index.npy`` (float64): so that two builds can be
  compared output for output.  The inputs depend only on the arguments.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

N_POINTS, NPOINT, RADIUS, NSAMPLE = 24000, 1024, 0.1, 32
MLP = [32, 32, 64]
METRIC = "sampled-points/sec (FPS+ballq+group-MLP, 24k-pt cloud)"
UNIT = "sampled points/s"
WORKLOAD = "pointnet++ SA1 forward: FPS 24000->1024, ball query r=0.1 K=32, group-MLP 9->[32,32,64], eval BN"
MLP_FLOP_PER_CLOUD = 2.0 * NPOINT * NSAMPLE * (9 * 32 + 32 * 32 + 32 * 64)      # SURVEY.md 8d: 0.220 GFLOP
B200_FP32_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12                                  # CUDA-core FMA peak at max clock
DUMP_CLOUDS = 128                     # 128 * (3 + 64) * 1024 * 4 bytes = 35 MB of dumped outputs at most


def host_cores() -> int:
    """Host threads this process may actually use (cgroup / affinity aware), not the machine total."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:   # cgroup v2 CPU quota
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        pass
    return n


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1590.0}, "fallback"


def ncu_constants():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_constants.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------ NUMA
def nvml_handle(local_gpu: int):
    """NVML handle of CUDA device ``local_gpu``: NVML enumerates every GPU of the machine and ignores CUDA_VISIBLE_DEVICES, so
    the entry of that variable (an index or a GPU-<uuid>) is translated first."""
    import pynvml
    pynvml.nvmlInit()
    vis = [e.strip() for e in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if e.strip()]
    if local_gpu < len(vis):
        e = vis[local_gpu]
        if e.isdigit():
            return pynvml.nvmlDeviceGetHandleByIndex(int(e))
        return pynvml.nvmlDeviceGetHandleByUUID(e if isinstance(e, bytes) else e.encode())
    return pynvml.nvmlDeviceGetHandleByIndex(local_gpu)


def sysfs_bdf(domain: int, bus: int, device: int) -> str:
    return f"{domain:04x}:{bus:02x}:{device:02x}.0"


def numa_bind(local_gpu: int, bdf: str = None) -> dict:
    """Bind this process (threads AND future page allocations, i.e. the pinned staging buffers) to the NUMA node of
    its GPU: CPU affinity from /sys/bus/pci/devices/<bdf>/numa_node, memory policy MPOL_PREFERRED through the raw
    set_mempolicy syscall (no libnuma in the image).  Must run before the host buffers are allocated.  ``bdf`` = the PCI
    address when the caller knows it (from CUDA); otherwise it is looked up through NVML."""
    info = {"gpu": local_gpu, "node": None, "cpus": None, "mempolicy": None}
    try:
        if bdf is None:
            import pynvml
            bus = pynvml.nvmlDeviceGetPciInfo(nvml_handle(local_gpu)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            bdf = bus.lower()
            if len(bdf.split(":")[0]) == 8:          # nvml prints an 8-digit domain, sysfs uses 4
                bdf = bdf[4:]
        info["pci"] = bdf
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return info
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info["cpus"] = f"{len(allowed)} cpus of node {node}"
        info["node"] = node
        libc = ctypes.CDLL(None, use_errno=True)
        mask = ctypes.c_ulong(1 << node)
        MPOL_PREFERRED, SYS_set_mempolicy = 1, 238          # x86_64
        rc = libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, ctypes.byref(mask), ctypes.c_ulong(8 * ctypes.sizeof(mask)))
        info["mempolicy"] = "preferred" if rc == 0 else f"errno {ctypes.get_errno()}"
    except Exception as e:      # best effort: a missing sysfs entry must not fail the bench
        info["error"] = repr(e)[:120]
    return info


class ClockSampler:
    """Samples SM clock and throttle reasons with NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = nvml_handle(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def make_clouds(rank: int, count: int, distinct: int = 8) -> torch.Tensor:
    """(count, 6, N) feature tensors [xyz; normal]; cloud j on rank r has seed 1000*r + (j mod distinct).
    To keep start-up short only ``distinct`` clouds are synthesised per rank and tiled; the FPS pruning rate is
    data-dependent, so ``config.distinct_clouds`` states it."""
    from toothgroupnetwork_b200 import clouds
    base = [clouds.arch_features(N_POINTS, clouds.cloud_seed(rank, j))[0] for j in range(min(count, distinct))]
    return torch.stack([base[j % len(base)] for j in range(count)]).contiguous()


def build_module(device):
    from toothgroupnetwork_b200 import pointnet2_utils as pn2
    torch.manual_seed(0)
    sa = pn2.PointNetSetAbstraction(NPOINT, RADIUS, NSAMPLE, 9, MLP, False)
    g = torch.Generator().manual_seed(1)
    with torch.no_grad():
        for bn in sa.mlp_bns:     # non-trivial eval statistics
            bn.running_mean.copy_(torch.randn(bn.running_mean.shape, generator=g) * 0.1)
            bn.running_var.copy_(torch.rand(bn.running_var.shape, generator=g) + 0.5)
    return sa.to(device).eval()


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_step(feats: torch.Tensor, sa_cpu_layers):
    """The oracle's port of the reference's CPU-capable formulation on ``feats`` (b,6,N), one cloud per OpenMP thread:
    torch-loop FPS with start 0 (pointnet2_utils.py:103-118), query_ball_point (:120-144), then gather +
    conv1x1+BN+ReLU x3 + max (:227-237) on cache-resident (K, C) tiles."""
    from oracle import oracle
    xyz = feats[:, :3].permute(0, 2, 1).contiguous().numpy()
    pts = feats.permute(0, 2, 1).contiguous().numpy()
    _, new_np, gi_np = oracle.sa_sample_and_search_batch(xyz, NPOINT, RADIUS, NSAMPLE)
    out = oracle.sa_group_mlp_max_batch(xyz, pts, new_np, gi_np, sa_cpu_layers)
    return torch.from_numpy(new_np), torch.from_numpy(out)


def cpu_layers_of(sa):
    from oracle import oracle
    out = []
    for c, b in zip(sa.mlp_convs, sa.mlp_bns):
        out.append(oracle.MlpParams(c.weight.detach().cpu().reshape(c.weight.shape[0], -1), c.bias.detach().cpu(),
                                    b.weight.detach().cpu(), b.bias.detach().cpu(), b.running_mean.detach().cpu(),
                                    b.running_var.detach().cpu(), b.eps))
    return out


def time_cpu(layers, sample_clouds: int, steps: int, warmup: int):
    cores = host_cores()
    torch.set_num_threads(cores)
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    feats = make_clouds(0, sample_clouds)
    for _ in range(warmup):
        cpu_reference_step(feats, layers)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(feats, layers)
    dt = (time.perf_counter() - t0) / steps
    return sample_clouds * NPOINT / dt, dt, cores


def dump_outputs(out_dir: str, new_xyz: torch.Tensor, new_points: torch.Tensor) -> None:
    """A fixed, seeded sample of the clouds of one step's outputs, as float32 .npy files (see the module docstring)."""
    B = new_xyz.shape[0]
    pick = np.sort(np.random.default_rng(0).choice(B, size=min(B, DUMP_CLOUDS), replace=False))
    index = torch.from_numpy(pick).to(new_xyz.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "new_xyz.npy"), new_xyz.index_select(0, index).float().cpu().numpy())
    np.save(os.path.join(out_dir, "new_points.npy"), new_points.index_select(0, index).float().cpu().numpy())
    np.save(os.path.join(out_dir, "cloud_index.npy"), pick.astype(np.float64))


def elementwise_rel(a: torch.Tensor, b: torch.Tensor, floor: float = 0.05) -> float:
    a, b = a.double(), b.double()
    return float(((a - b).abs() / b.abs().clamp(min=floor * float(b.abs().max()) + 1e-300)).max())


# ------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clouds", type=int, default=1184, help="clouds per GPU per step (8 per SM)")
    ap.add_argument("--cpu-clouds", type=int, default=0, help="clouds in the CPU sample (default: 2 per host core, at most 64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the ref_gpu / latency / kNN / C1 legs (profiling runs)")
    ap.add_argument("--no-numa", action="store_true")
    ap.add_argument("--e2e-chunk", type=int, default=148, help="clouds per pipelined chunk of the end-to-end measurement")
    ap.add_argument("--e2e-streams", type=int, default=2)
    ap.add_argument("--e2e-groups", default="1", help="chunks per compute group of the end-to-end pipeline")
    ap.add_argument("--e2e-sa-engine", type=int, default=None, help="group-MLP engine inside the end-to-end pipeline (5: half-size CTAs that co-reside with other chunks' kernels)")
    ap.add_argument("--e2e-fps-mode", type=int, default=None, help="FPS shape of every pipelined chunk (-14: 4 warps per cloud, -18: 8, -26: 16); default: by clouds in flight")
    ap.add_argument("--fps-mode", type=int, default=0, help="0 auto; 100*G+CS resident shape, -2 bucket, -(10+W) bucket with W warps per cloud (experiments)")
    ap.add_argument("--ball-path", type=int, default=0, help="0 auto, 4 index-order tile scan, 8 uniform grid (experiments)")
    ap.add_argument("--sa-engine", type=int, default=0, help="0 auto, 1 fp32 CUDA cores, 2 tcgen05 (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's outputs to DIR as .npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    from toothgroupnetwork_b200 import sharding
    rank, world, local = sharding.env_rank_world()
    config = {"workload": WORKLOAD, "clouds_per_gpu": args.clouds, "points_per_cloud": N_POINTS, "npoint": NPOINT,
              "radius": RADIUS, "nsample": NSAMPLE, "mlp": MLP, "parallelism": f"mesh-sharded x{world}",
              "l2": "inputs larger than L2, no flush", "distinct_clouds": min(args.clouds, 8),
              "data_note": "8 distinct synthetic clouds per rank, tiled: FPS pruning efficiency is data-dependent"}

    if args.impl == "reference":
        # Reference arm: CPU, rank 0 only, bounded sample of the same workload.
        if rank != 0:
            return
        sa = build_module("cpu")
        cores = host_cores()
        sample = args.cpu_clouds or min(64, 2 * cores)
        value, dt, cores = time_cpu(cpu_layers_of(sa), sample, max(1, args.steps), max(0, args.warmup))
        line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"{sample} clouds of {N_POINTS} points per step (one cloud per host thread, {cores} threads)"},
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU path)")
    numa = {"bound": False} if args.no_numa else numa_bind(local)
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if not args.no_numa:
        # CUDA's own answer for this device; if the NVML lookup above named another GPU (a remapped device list), bind again --
        # the pinned staging buffers are allocated further down
        props = torch.cuda.get_device_properties(local)
        bdf = sysfs_bdf(props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        if numa.get("pci") != bdf:
            numa = dict(numa_bind(local, bdf), rebound_from=numa.get("pci"))
    rank, world, local = sharding.init("nccl")
    from toothgroupnetwork_b200 import _lib as L
    from toothgroupnetwork_b200 import pointnet2_utils as pn2

    sa = build_module(device)
    pn2.set_sa_engine(args.sa_engine)
    pn2.set_ball_path(args.ball_path)
    pn2.set_fps_mode(args.fps_mode)
    B = args.clouds
    host_feats = make_clouds(rank, B).pin_memory()
    feats = host_feats.to(device)
    xyz = feats[:, :3].contiguous()
    folded = sa._folded.update(sa.mlp_convs, sa.mlp_bns)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def staged_step(events=None):
        """Same kernels as sa.forward, with events between the three stages."""
        xyz_t = pn2.transpose_last2(xyz)
        feats_t = pn2.transpose_last2(feats)
        if events: events[0].record()
        fps = pn2._fps_batched(xyz_t, NPOINT)
        if events: events[1].record()
        new_xyz_t = pn2._take_rows(xyz_t.view(-1, 3), fps).view(B, NPOINT, 3)
        gidx = pn2._ball_query(RADIUS, NSAMPLE, xyz_t, new_xyz_t, False, None, 1)
        if events: events[2].record()
        out = torch.empty((B, MLP[-1], NPOINT), dtype=torch.float32, device=device)
        pn2.sa_group_mlp_max(xyz_t, feats_t, new_xyz_t, gidx, True, folded, out, 0)
        if events: events[3].record()
        return new_xyz_t.permute(0, 2, 1), out

    # -------- parity on this rank: (a) public module == staged kernels, (b) cloud 0 against the CPU oracle -------------
    with torch.no_grad():
        a = staged_step()
        b = sa(xyz, feats)
        staged_equal = bool(torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]))
        pn2.set_reference_device("cpu")                      # the checker restates the reference on CPU tensors
        one = sa(xyz[:1].contiguous(), feats[:1].contiguous())
        pn2.set_reference_device("cuda")
    from oracle import oracle
    want_xyz, want_pts = oracle.set_abstraction(host_feats[:1, :3].contiguous(), host_feats[:1].contiguous(), NPOINT, RADIUS, NSAMPLE,
                                                cpu_layers_of(sa))      # CPU restatement: pointops FPS, query_ball_point, conv/BN/ReLU/max
    oracle_xyz_bitwise = bool(torch.equal(one[0].cpu(), want_xyz))
    oracle_rel = elementwise_rel(one[1].cpu(), want_pts)
    parity_ok = staged_equal and oracle_xyz_bitwise and oracle_rel < 1e-4

    # -------- device-resident timing of the public module call ---------------------------------------------------------
    with torch.no_grad():
        for _ in range(args.warmup):
            sa(xyz, feats)
        t_start, t_end = ev(), ev()
        sharding.barrier()
        torch.cuda.synchronize()
        launches0 = L.launch_count()
        with ClockSampler(local) as clk:
            t_start.record()
            for s in range(args.steps):
                last = sa(xyz, feats)
            t_end.record()
            torch.cuda.synchronize()
        launches = L.launch_count() - launches0
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, *last)
        del last
        sharding.barrier()
        # stage breakdown: the same kernels with events between the stages (not part of `value`)
        stage_events = [[ev() for _ in range(4)] for _ in range(min(args.steps, 5))]
        for e in stage_events:
            staged_step(e)
        torch.cuda.synchronize()
    local_s = t_start.elapsed_time(t_end) / 1e3
    total_s = sharding.max_over_ranks(local_s, device)
    fps_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in stage_events]))
    ball_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in stage_events]))
    mlp_ms = float(np.mean([e[2].elapsed_time(e[3]) for e in stage_events]))
    value = world * B * NPOINT * args.steps / total_s

    # -------- end to end through the public API with host buffers -----------------------------------
    out_xyz_host = torch.empty((B, 3, NPOINT), dtype=torch.float32).pin_memory()
    out_pts_host = torch.empty((B, MLP[-1], NPOINT), dtype=torch.float32).pin_memory()

    from toothgroupnetwork_b200.pipeline import HostPipeline
    pipe = HostPipeline(sa, chunk_clouds=args.e2e_chunk, n_streams=args.e2e_streams,
                        groups=[int(g) for g in args.e2e_groups.split(",")], fps_mode=args.e2e_fps_mode, sa_engine=args.e2e_sa_engine)

    def e2e_step():
        # public API on host buffers, one batch at a time: chunks of the batch go H2D -> module.forward -> D2H on a few
        # streams, so copies overlap kernels WITHIN the batch (every byte still crosses PCIe inside the timed region)
        pipe(host_feats, out_xyz_host, out_pts_host)

    def timed(fn, after=None):
        with torch.no_grad():
            for _ in range(args.warmup):
                fn()
            if after:
                after()
            t0, t1 = ev(), ev()
            sharding.barrier()
            torch.cuda.synchronize()
            t0.record()
            for _ in range(args.steps):
                fn()
            if after:
                after()
            t1.record()
            torch.cuda.synchronize()
            sharding.barrier()
        return t0.elapsed_time(t1) / 1e3

    chunked_s = timed(e2e_step)
    chunked_xyz, chunked_pts = out_xyz_host.clone(), out_pts_host.clone()
    out_xyz_host.zero_()
    out_pts_host.zero_()
    # a stream of batches through the same public object: submit() queues a whole batch and returns, so the H2D copy of batch
    # i+1 overlaps the kernels of batch i and the D2H of batch i-1 (two device input buffers); every step's input still goes
    # host -> device and every step's result device -> host inside the timed region, drain() included
    stream_s = timed(lambda: pipe.submit(host_feats, out_xyz_host, out_pts_host), after=pipe.drain)
    stream_equal = bool(torch.equal(out_xyz_host, chunked_xyz) and torch.equal(out_pts_host, chunked_pts))
    e2e_mode = "stream of batches (submit/drain)" if (stream_equal and stream_s < chunked_s) else "one batch at a time (chunked)"
    e2e_local_s = min(stream_s, chunked_s) if stream_equal else chunked_s
    e2e_modes_ms = {"one_batch_at_a_time_chunked": chunked_s * 1e3 / args.steps, "stream_of_batches": stream_s * 1e3 / args.steps,
                    "stream_results_equal_chunked": stream_equal}
    e2e_s = sharding.max_over_ranks(e2e_local_s, device)
    e2e_value = world * B * NPOINT * args.steps / e2e_s

    # -------- the one collective of the run: per-rank metric records ----------------------------------
    records = sharding.gather_metrics({"sampled_points": B * NPOINT * args.steps, "clouds": B * args.steps, "seconds": local_s,
                                       "parity_ok": float(parity_ok), "launches": launches,
                                       "numa_node": float(numa["node"]) if numa.get("node") is not None else -1.0,
                                       "e2e_seconds": e2e_local_s}, device)
    agg = sharding.reduce_metrics(records)

    if rank != 0:
        return
    peaks, peak_kind = measured_peaks()
    ncu = ncu_constants()
    fps_alg_bytes = 20.0 * (NPOINT - 1) * N_POINTS * B            # per FPS launch (SURVEY.md 8d)
    fps_compulsory = (12.0 * N_POINTS + 4.0 * NPOINT) * B
    fps_traffic = ncu.get("fps_dram_bytes_per_cloud", 0.0) * B or None
    fps_dram_gbs = fps_traffic / (fps_ms * 1e-3) / 1e9 if fps_traffic else None
    tensor_peak = peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops"))
    mlp_tflops = MLP_FLOP_PER_CLOUD * B / (mlp_ms * 1e-3) / 1e12
    ball_tflops = 8.0 * NPOINT * N_POINTS * B / (ball_ms * 1e-3) / 1e12
    stages = [
        {"stage": "fps", "kernel": "fps_bucket_sort_kernel + fps_bucket_kernel", "bound": "hbm (latency of the per-sample dependent chain in practice)",
         "ms": fps_ms, "compulsory_bytes": fps_compulsory, "traffic_bytes": fps_traffic, "traffic_over_compulsory": (fps_traffic / fps_compulsory) if fps_traffic else None,
         "achieved": fps_dram_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": (fps_dram_gbs / peaks["hbm_gbs"]) if fps_dram_gbs else None,
         "algorithmic_bytes": fps_alg_bytes, "algorithmic_gbs": fps_alg_bytes / (fps_ms * 1e-3) / 1e9,
         "traffic_source": ncu.get("fps_source"), "traffic_is": "constant from the committed ncu capture, scaled per cloud (not measured live)",
         "note": "the exact bucket pruning skips ~97% of the brute-force point-updates, so algorithmic_gbs exceeds the HBM peak by construction; frac is real DRAM traffic / time / peak"},
        {"stage": "ball_query", "kernel": "ball_query_kernel (index-order tile scan at r=0.1)", "bound": "fp32 issue", "ms": ball_ms,
         "achieved": ncu.get("ball_query_issue_active_pct"), "peak": 100.0, "unit": "% issue slots active (ncu, committed capture)",
         "frac": (ncu.get("ball_query_issue_active_pct") or 0.0) / 100.0, "source": ncu.get("ball_query_source"),
         "bruteforce_equivalent_tflops": ball_tflops, "fp32_peak_tflops": B200_FP32_TFLOPS,
         "note": "8*S*N FLOP per cloud / time exceeds the fp32 peak because the index-order scan stops after K hits; the bound that applies is instruction issue"},
        {"stage": "group_mlp", "kernel": "sa_mlp_tc_kernel (tcgen05 3xTF32)", "bound": "tensor", "ms": mlp_ms, "achieved": mlp_tflops, "peak": tensor_peak,
         "unit": "TFLOP/s useful (2*S*K*sum C_l*C_l+1)", "frac": mlp_tflops / tensor_peak, "peak_name": "bf16_tflops_sustained",
         "executed_over_useful_mma": ncu.get("group_mlp_executed_over_useful_mma"), "tensor_pipe_pct": ncu.get("group_mlp_tensor_pipe_pct"),
         "source": ncu.get("group_mlp_source")},
    ]
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config,
        "stage_ms": {"fps": fps_ms, "ball_query": ball_ms, "group_mlp": mlp_ms},
        "roofline": {"kernel": "fps_bucket_kernel (+ its sort prologue; one event pair brackets both)", "bound": "hbm",
                     "achieved": fps_dram_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": stages[0]["frac"],
                     "traffic": fps_traffic, "peak_kind": peak_kind, "compulsory_bytes": fps_compulsory,
                     "note": "achieved = DRAM bytes of the launch pair (ncu, committed capture) / live CUDA-event time; the SURVEY 8d "
                             "algorithmic figure (20*(M-1)*N bytes per cloud) is in roofline_stages[0].algorithmic_gbs and is not a bandwidth"},
        "roofline_stages": stages,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(host_feats.numel() * 4),
                "d2h_bytes_per_step": int((out_xyz_host.numel() + out_pts_host.numel()) * 4), "mode": e2e_mode, "ms_per_step_by_mode": e2e_modes_ms},
        "gpu_launches": int(agg["launches"]),
        "clocks": clk.summary(),
        "numa": dict(numa, per_rank_node=[int(r["numa_node"]) for r in records],
                     per_rank_e2e_ms_per_step=[round(r["e2e_seconds"] * 1e3 / args.steps, 3) for r in records]),
        "parity_ok": bool(agg["parity_ok"]),
        "parity": {"staged_kernels_equal_public_module": staged_equal, "cloud0_new_xyz_bitwise_vs_oracle": oracle_xyz_bitwise,
                   "cloud0_features_elementwise_rel_vs_oracle": oracle_rel, "floor": "0.05 * max|ref|", "tol": 1e-4},
    }
    if not args.no_extras:
        try:
            line.update(extras(device))
        except Exception as e:          # the extra legs must never take the headline line down with them
            line["extras_error"] = repr(e)[:300]
    if not args.no_cpu_baseline:
        cores = host_cores()
        sample = args.cpu_clouds or min(64, 2 * cores)
        cv, cdt, cores = time_cpu(cpu_layers_of(sa.cpu()), sample, 2, 1)
        line["cpu_baseline"] = {"value": cv, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"{sample} clouds of {N_POINTS} points per step (one cloud per host thread, {cores} threads), 2 timed steps"}
    print(json.dumps(line))


def extras(device) -> dict:
    """Rank-0 legs beside the headline: reference GPU path, latency table, C1, kNN mix (scripts/op_bench.py)."""
    import op_bench
    out = {}
    with torch.no_grad():
        rows = op_bench.fps_latency_table(batches=(1, 16, 148, 1184), npoints=(1024, 4096), with_ref=op_bench.ref_available())
        out["latency_ms"] = {"fps": rows}
        c1 = next(r for r in rows if r["clouds"] == 1 and r["m"] == 4096)
        out["c1"] = dict(c1, config="BASELINE configs[0]: furthest_point_sample 24000->4096 on one cloud", **op_bench.c1_parity())
        out["knn"] = op_bench.knn_table(with_ref=op_bench.ref_available())
        if op_bench.ref_available() and op_bench.ref_models_available():
            out["ref_gpu"] = {"what": "the reference's own GPU path for the bench step (verbatim FPS kernel + reference torch ball query / "
                                      "gather / Conv2d+BN+ReLU / max, IEEE fp32 convolutions), CUDA events, same GPU",
                              "runs": [op_bench.ref_gpu_step(Bc, False) for Bc in (1, 16)]}
            out["latency_ms"]["sa1_step"] = [{k: r[k] for k in ("clouds", "ours_ms", "ref_gpu_ms", "speedup")} for r in out["ref_gpu"]["runs"]]
        else:
            out["ref_gpu"] = {"unavailable": "oracle/_ref (reference kernels / python snapshot) not present on this box"}
        # SURVEY 8(f) rows built after the hot path: each leg is independent and may not take the bench line down with it
        nxt = {}
        for name, leg in (("raw_mesh_fps_100k_to_24k", op_bench.raw_mesh_fps), ("dbscan_moved_foreground", op_bench.dbscan_row),
                          ("tgnet_fps_nograd_forward", op_bench.tgnet_nograd_row)):
            if name == "tgnet_fps_nograd_forward" and not (op_bench.ref_available() and op_bench.ref_models_available()):
                nxt[name] = {"unavailable": "reference python snapshot not present on this box"}
                continue
            try:
                nxt[name] = leg()
            except Exception as e:                                   # noqa: BLE001 -- reported, not hidden
                nxt[name] = {"error": repr(e)[:300]}
        out["next_rows"] = nxt
    return out


if __name__ == "__main__":
    try:
        main()
    finally:
        import torch.distributed as _dist
        if _dist.is_available() and _dist.is_initialized():
            _dist.destroy_process_group()
