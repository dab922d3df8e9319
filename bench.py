#!/usr/bin/env python
"""bench.py — headline benchmark of the CRFConv hot path (BASELINE.json metric: CRFConv fwd+bwd points/s at N=40,960, k=16).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config S1|C3|C4|C5] [--clouds B] [--impl reference] [--dump-outputs DIR]

--config S1 (default; SURVEY.md §8 S1 = BASELINE configs[0] shape on the GPU): one *step* = forward + backward of ONE
``ContinuousGaussianCRFConv(128, 64, 64, steps=1)`` layer (N=40,960 points, Nc=10,240 coarse points, K=16, Cu=128, Cp=Co=64,
hidden F=16) over a batch of B = 6 synthetic S3DIS-room-shaped clouds per GPU.
--config C3 / C4 / C5 (BASELINE configs[2..4]): one step = forward + cross-entropy + backward of the whole ``PointConvResNet``
(6 input channels, use_crf=True) on B clouds per GPU of 40,960 points / 13 classes (C3, B=6), 45,056 points / 19 classes
(C4, SemanticKITTI-shaped, B=8) or 65,536 points / 8 classes (C5, Semantic3D-shaped, B=2); the 5-level kNN pyramid is an input.
Clouds are independent ⇒ ranks hold different clouds (weak scaling); the only exchange is the NCCL all-reduce of the flat fp32
parameter gradient, inside the timed step when N > 1.

value        : points/s with inputs resident in HBM (CUDA-event timed, max over ranks), the step replayed as a CUDA graph.
e2e          : same metric through the public API with HOST (pinned) inputs: H2D of every input of the step (S1: unary / pairwise /
               up_idx / neighbor_idx; C3-C5: points, features, labels — the pyramid is then built on the GPU inside the timed
               region) and a D2H read of the loss every step.  Ranks bind to their GPU's NUMA node before allocating pinned memory;
               `e2e.h2d_gbs_per_gpu` and `e2e.h2d_probe_gbs_per_gpu` (all ranks copying at once, no compute) locate the host-side ceiling.
               S1: the inputs go through `crfconv_b200.host_io.HostStager`; with --pack-index on the int64 index tensors are narrowed
               to 16 bits on the host (every step, inside the timed region), copied packed and widened on the device; `auto`
               (default) times both forms for 8 steps each and runs the timed region with the faster one (`e2e.index_packing`).
               `h2d_bytes_per_step` counts the bytes actually copied, `h2d_bytes_reference_format` the int64 form.
roofline     : the WHOLE step against SURVEY.md §8(d)'s algorithmic bytes (S1: 79,298,560 B per cloud fwd+bwd; C3-C5: the shape
               walker `network_algo_bytes`) — `frac` is the north_star fraction.  `roofline.dominant_kernel` names the single
               kernel with the largest share of the step; `kernels` lists every kernel call with its own bytes and GB/s.
cpu_baseline / --impl reference: the CPU port of the reference (oracle/layers.py, PyTorch CPU, all host threads) on the SAME
               workload (S1: the same 6 clouds per step; C3-C5: a bounded 2-cloud sample).  The reference itself is Python and is
               not present on the GPU box.
--dump-outputs DIR: after the timed steps, rank 0 writes what the last timed step returned to its caller as DIR/<name>.npy (float32),
               so that two builds can be compared output for output on the same seeded inputs.  S1: `out` and `grad_unary` /
               `grad_pairwise` (a fixed sample of 32,768 of the B x 40,960 point rows, 8,192 of the B x 10,240 coarse rows of
               `grad_unary`: ≈21 MB whatever B; `out_rows` / `grad_unary_rows` are the sampled row indices into the flattened
               batch); C3-C5: `loss`.  Both: `grad_params`, the flat fp32 parameter gradient that the step hands to the
               all-reduce / optimiser (parameters in `module.parameters()` order).  With N > 1 GPUs only rank 0 writes (its own
               clouds).  Several kernels accumulate with atomics, so two runs of one build agree to fp32 rounding, not bit for bit:
               compare with a tolerance relative to each array's scale (a gradient that is zero in exact arithmetic, such as the
               bias of a BatchNorm that feeds another batch-statistics BatchNorm, is rounding noise on its own).
--steps K    : the number of timed steps of every timed loop (the headline, the e2e arm and --impl reference).  The reference arm
               runs K full fwd+bwd passes on the CPU (S1: 6 x 40,960 points, seconds each): pass a small K there.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POINTS, K_NBR, CU, CP, RATIO = 40960, 16, 128, 64, 4
ALGO_BYTES_PER_CLOUD = 4 * (2 * N_POINTS * CP + 3 * (N_POINTS // RATIO) * CU + 3 * N_POINTS * CP) + 16 * N_POINTS * (K_NBR + 1)  # 79,298,560
L2_BYTES = 126 * 2**20
METRIC = "CRFConv fwd+bwd points/s (N=40960,k=16)"

# BASELINE.json configs[2..4]: the full segmentation network (in_channels = 6: xyz + rgb, trainval.py:33-35,61)
NET_CONFIGS = {
    "C3": {"points": 40960, "classes": 13, "clouds": 6, "name": "S3DIS-shaped batch of 6 x 40,960 points, 13 classes (BASELINE configs[2])"},
    "C4": {"points": 45056, "classes": 19, "clouds": 8, "name": "SemanticKITTI-shaped scans, 45,056 points, 19 classes, 8 clouds per GPU (BASELINE configs[3])"},
    "C5": {"points": 65536, "classes": 8, "clouds": 2, "name": "Semantic3D-shaped crops, 65,536 points, 8 classes, 2 clouds per GPU (BASELINE configs[4])"},
}


def crf_layer_algo_bytes(N, Nc, Cu, Cp, Co, K=16):
    """SURVEY.md §8(d): every API-boundary tensor crosses HBM once per pass; fwd+bwd of one dense CRF layer, per cloud."""
    return 4 * (2 * N * Co + 3 * Nc * Cu + 3 * N * Cp) + 16 * N * (K + 1)


def network_algo_bytes(N0, n_classes, in_channels=6, K=16):
    """Shape walker over PointConvResNet (models/point_conv_big.py:110-167) with SURVEY.md §8(d)'s per-layer formulas: fwd+bwd
    algorithmic bytes per cloud = 10 ResNetBBlocks + 4 CRF layers + classifier (hidden activations excluded: they may be recomputed)."""
    ratios = (4, 4, 4, 4, 2)
    Ns = [N0]
    for r in ratios[:4]:
        Ns.append(Ns[-1] // r)
    C = [32, 64, 128, 256, 512]

    def block(n_in, n_out, cin, cout):
        return 4 * n_in * 3 * cin + 4 * n_out * 2 * cout + 2 * (12 * (n_in + n_out) + 8 * n_out * K)
    total = block(Ns[0], Ns[0], in_channels, C[0]) + block(Ns[0], Ns[0], C[0], C[0])
    for l in range(1, 5):
        total += block(Ns[l - 1], Ns[l], C[l - 1], C[l]) + block(Ns[l], Ns[l], C[l], C[l])
    for l in (3, 2, 1, 0):                                 # deconv4..deconv1: unary = level l+1 (C[l+1]), pairwise = skip at level l (C[l])
        total += crf_layer_algo_bytes(Ns[l], Ns[l + 1], C[l + 1], C[l], C[l], K)
    total += 4 * Ns[0] * (3 * C[0] + 2 * n_classes)        # classifier: x read (fwd, bwd) + dx written, logits written + their gradient read
    return total


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        time.sleep(0.05)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def bind_to_gpu_numa_node(torch, local_rank):
    """Pins this process to the CPUs of its GPU's NUMA node and prefers that node's memory BEFORE any pinned allocation, so that
    each rank's H2D copies read local DRAM instead of crossing the socket interconnect.  Returns a description for the bench line."""
    info = {"numa_node": None, "cpus": None, "mempolicy": None}
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        info["pci"] = bus
        if node < 0:
            info["numa_node"] = -1
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        info["numa_node"], info["cpus"] = node, len(cpus)
        try:                                            # set_mempolicy(MPOL_PREFERRED = 1, nodemask, maxnode): x86_64 syscall 238
            mask = (ctypes.c_ulong * 16)()
            mask[node // 64] = 1 << (node % 64)
            rc = ctypes.CDLL(None, use_errno=True).syscall(238, 1, mask, 16 * 64)
            info["mempolicy"] = "preferred" if rc == 0 else f"errno {ctypes.get_errno()}"
        except Exception as exc:                         # noqa: BLE001
            info["mempolicy"] = f"unavailable ({type(exc).__name__})"
    except Exception as exc:                             # noqa: BLE001
        info["error"] = f"{type(exc).__name__}: {exc}"[:120]
    return info


def h2d_probe(torch, dev, host_tensors, barrier, reps=8):
    """H2D bandwidth of this rank's pinned input set with every rank copying at the same time and no compute: the host-side ceiling."""
    dst = {k: torch.empty_like(v, device=dev) for k, v in host_tensors.items()}
    nbytes = sum(v.numel() * v.element_size() for v in host_tensors.values())
    for k, v in host_tensors.items():
        dst[k].copy_(v, non_blocking=True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for k, v in host_tensors.items():
            dst[k].copy_(v, non_blocking=True)
    e1.record()
    barrier()
    return reps * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_layer_points_per_s(clouds=6, repeats=4, warm=1):
    """Reference layer restated on CPU (oracle/layers.py) fwd+bwd; kNN indices from the compiled reference when shipped."""
    import torch
    from oracle import layers as ol
    from oracle import native as on
    from oracle import synthetic
    torch.set_num_threads(os.cpu_count() or 1)
    knn = (lambda s, q, k: on.ref_knn_batch(s, q, k, omp=True)) if on.have_ref_knn() else on.knn_batch
    n = N_POINTS
    inp = synthetic.crf_layer_inputs(clouds, n, K_NBR, CU, CP, RATIO, seed=0, knn_batch_fn=knn)
    torch.manual_seed(0)
    layer = ol.ContinuousGaussianCRFConv(CU, CP, CP, steps=1).train()
    u, p = inp.unary.requires_grad_(True), inp.pairwise.requires_grad_(True)
    ts = []
    for i in range(warm + repeats):
        t0 = time.perf_counter()
        out = layer(u, p, inp.up_idx, inp.neighbor_idx)
        out.sum().backward()
        dt = time.perf_counter() - t0
        if i >= warm:
            ts.append(dt)
        layer.zero_grad(); u.grad = None; p.grad = None
    t = statistics.median(ts)
    return clouds * n / t, t, {"value": clouds * n / t, "unit": "points/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": f"{clouds} clouds x {n} points (the GPU arm's step), CRF layer fwd+bwd, median of {repeats} after {warm} "
                                         f"warm-up (oracle/layers.py on torch CPU, {torch.get_num_threads()} threads)"}


def cpu_network_points_per_s(cfg, clouds=2, repeats=2, warm=1):
    """Reference network restated on CPU (oracle/layers.py PointConvResNet) fwd + cross-entropy + bwd on a bounded sample."""
    import types
    import torch
    import torch.nn.functional as Fn
    from oracle import layers as ol
    from oracle import native as on
    from oracle import synthetic
    torch.set_num_threads(os.cpu_count() or 1)
    knn = (lambda s, q, k: on.ref_knn_batch(s, q, k, omp=True)) if on.have_ref_knn() else on.knn_batch
    n, ncls = cfg["points"], cfg["classes"]
    pos = synthetic.room_cloud(clouds, n, seed=0)
    ms = synthetic.build_multiscale(pos, knn)
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.from_numpy(pos), torch.rand(clouds, n, 3, generator=g)], -1)
    y = torch.randint(0, ncls, (clouds * n,), generator=g)
    torch.manual_seed(0)
    net = ol.PointConvResNet(6, ncls).train()
    data = types.SimpleNamespace(x=x, multiscale=ms)
    ts = []
    for i in range(warm + repeats):
        t0 = time.perf_counter()
        Fn.cross_entropy(net(data), y).backward()
        dt = time.perf_counter() - t0
        if i >= warm:
            ts.append(dt)
        net.zero_grad()
    t = statistics.median(ts)
    return clouds * n / t, t, {"value": clouds * n / t, "unit": "points/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": f"{clouds} clouds x {n} points, PointConvResNet fwd + CE + bwd, median of {repeats} after {warm} warm-up "
                                         f"(oracle/layers.py on torch CPU, {torch.get_num_threads()} threads; pyramid prebuilt)"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    steps = args.steps
    if args.config == "S1":
        v, t, cb = cpu_layer_points_per_s(clouds=args.clouds or 6, repeats=steps, warm=min(max(args.warmup, 1), 2))
        workload = (f"single ContinuousGaussianCRFConv(128,64,64,steps=1) fwd+bwd, N=40960, Nc=10240, K=16, {args.clouds or 6} clouds per step "
                    "(the same step as the GPU arm)")
        metric = METRIC
    else:
        cfg = NET_CONFIGS[args.config]
        v, t, cb = cpu_network_points_per_s(cfg, clouds=2, repeats=steps, warm=1)
        workload = f"PointConvResNet(6,{cfg['classes']},use_crf=True) fwd+CE+bwd, {cfg['name']}; CPU arm: 2 clouds per step (bounded sample)"
        metric = "PointConvResNet fwd+bwd points/s"
    line = {"impl": "reference", "metric": metric, "value": v, "unit": "points/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": workload, "config": args.config},
            "cpu_baseline": cb, "e2e": {"value": v, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def make_inputs(torch, B, dev, seed):
    from crfconv_b200 import nearest_neighbors as nn_
    g = torch.Generator(device="cpu").manual_seed(seed)
    pos = (torch.rand(B, N_POINTS, 3, generator=g) * torch.tensor([8.0, 6.0, 3.0])).to(dev)
    nbr = nn_.knn_batch(pos, pos, K_NBR)
    choice = torch.randperm(N_POINTS, generator=g)[: N_POINTS // RATIO].to(dev)
    up = nn_.knn_batch(pos[:, choice].contiguous(), pos, 1)
    unary = torch.randn(B, N_POINTS // RATIO, CU, generator=g).to(dev)
    pair = torch.randn(B, N_POINTS, CP, generator=g).to(dev)
    return {"pos": pos, "unary": unary, "pairwise": pair, "up_idx": up, "neighbor_idx": nbr}


def _single_kernel_name(call):
    """C-ABI call label of ops.profile_calls → the CUDA kernel(s) it launches (for `roofline.dominant_kernel`)."""
    table = {"crf_step_bwd_fused": "cl::step_bwd_kernel", "crf_step_fwd[16]": "mf::step_fwd_kernel<16>", "out16_bwd": "cl::out_bwd_kernel",
             "linear_fwd_bn[128->64]": "lin3::fwd3_kernel<64>", "up16_fwd[64]": "cl::up16_fwd_kernel<64>",
             "linear_bwd[64<-128]:dgrad": "lin3d::dgrad3_kernel<128>", "linear_bwd[64<-128]:wgrad": "lin3w::wgrad3_kernel<64>", "bn_bwd_reduce_fin[64]": "lin::bn_bwd_reduce_kernel",
             "mid16_bwd": "cl::mid16_bwd_kernel", "lin16_fwd[64]": "cl::lin16_fwd_kernel<64>", "lin16_fwd[128]": "cl::lin16_fwd_kernel<128>",
             "lin16_fwd[16]": "cl::lin16_fwd_kernel<16>", "in16_dgrad[64]": "cl::in16_dgrad_kernel<64>", "in16_wgrad[64]": "cl::in16_wgrad_kernel<64>"}
    return table.get(call, call)


def _timed(torch, dist, world, dev, step, steps, barrier):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms



def warm_up(torch, dist, world, dev, step, min_steps, min_seconds=0.5, chunk=8):
    """Untimed warm-up: at least `min_steps` steps and `min_seconds` of load (so that nvidia-smi samples land under load).  The
    number of steps must be the SAME on every rank — a step contains the gradient all-reduce, and ranks that stop on their own
    clocks would issue different numbers of collectives (a hang waiting for the NCCL watchdog).  Rank 0's clock decides, chunk by
    chunk, and the decision is broadcast."""
    t_w = time.perf_counter()
    i = 0
    while True:
        for _ in range(chunk):
            step(i)
            i += 1
        torch.cuda.synchronize()
        more = i < min_steps or time.perf_counter() - t_w < min_seconds
        if world > 1:
            flag = torch.tensor([1 if more else 0], device=dev, dtype=torch.int32)
            dist.broadcast(flag, 0)
            more = bool(int(flag.item()))
        if not more:
            return i

def _ncu_traffic(name):
    """DRAM bytes (read + write) of one step from the committed ncu capture (profiles/ncu_r02_metrics.json), or None."""
    try:
        met = json.load(open(os.path.join(ROOT, "profiles", "ncu_r02_metrics.json")))
        return met.get(name)
    except Exception:
        return None


def sample_rows(torch, n, keep, dev):
    """Sorted fixed sample of `keep` of `n` rows (its own seeded generator: the same rows in every run)."""
    return torch.randperm(n, generator=torch.Generator(device="cpu").manual_seed(0))[:keep].sort().values.to(dev)


def dump_outputs(path, arrays):
    """Writes every tensor of `arrays` as <path>/<name>.npy in float32."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().float().cpu().numpy())


def run_gpu(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: crfconv_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)          # before the first pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if args.config != "S1":
        return run_gpu_network(args, rank, local_rank, world, dev, numa)
    from crfconv_b200 import ops
    from crfconv_b200.continuous_crf_conv_big import ContinuousGaussianCRFConv
    from crfconv_b200 import nearest_neighbors as nn_

    B = args.clouds or 6
    torch.manual_seed(1234)
    layer = ContinuousGaussianCRFConv(CU, CP, CP, steps=1).to(dev).train()
    with torch.no_grad():
        layer.c.add_(0.1 * torch.randn_like(layer.c))
    from crfconv_b200.distributed import FlatGradients
    # bind=False: autograd adopts the gradient tensors the fused layer returns — views of ONE flat allocation — so there is no
    # accumulate kernel per parameter, and the all-reduce runs in place on that allocation (one collective, no copies)
    fg = FlatGradients(layer, bind=False)

    in_bytes = B * (4 * ((N_POINTS // RATIO) * CU + N_POINTS * CP) + 8 * N_POINTS * (K_NBR + 1))
    nsets = max(2, -(-2 * L2_BYTES // max(in_bytes, 1)))     # rotate enough input sets that a step never finds its inputs in L2
    nsets = min(nsets, 8)
    sets = [make_inputs(torch, B, dev, seed=100 * rank + s) for s in range(nsets)]
    for s in sets:
        s["unary"].requires_grad_(True)
        s["pairwise"].requires_grad_(True)
    cot = torch.ones(B, N_POINTS, CP, device=dev)
    # --dump-outputs: input set -> what a step on it returns to the caller (a replayed graph overwrites the tensors of its capture)
    results = {}

    def keep(k, out, s):
        if args.dump_outputs:
            results[k] = {"out": out, "grad_unary": s["unary"].grad, "grad_pairwise": s["pairwise"].grad,
                          "grad_params": [p.grad for p in fg.params]}

    def eager_step(i, reduce=True):
        s = sets[i % nsets]
        fg.zero()
        out = layer(s["unary"], s["pairwise"], s["up_idx"], s["neighbor_idx"])
        out.backward(cot)
        if reduce:
            fg.all_reduce()                       # no-op at world == 1
        keep(i % nsets, out, s)
        s["unary"].grad = None
        s["pairwise"].grad = None

    # The kernel launches of one fwd+bwd are captured ONCE per input set into a CUDA graph and replayed: with < 1 ms of GPU work
    # per step the Python/ctypes launch path (≈1.8 ms per step) would otherwise be the bottleneck.  The gradient all-reduce
    # (ReduceOp.AVG: no separate scaling kernel) stays outside the graph.
    graphs, launches_per_step = [], 0
    if args.graph:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i in range(3):
                eager_step(i)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for k in range(nsets):
            s = sets[k]
            g = torch.cuda.CUDAGraph()
            ops.COUNTERS["launches"] = 0
            with torch.cuda.graph(g):
                fg.zero()
                out = layer(s["unary"], s["pairwise"], s["up_idx"], s["neighbor_idx"])
                out.backward(cot)
            launches_per_step = ops.COUNTERS["launches"]
            keep(k, out, s)
            s["unary"].grad = None
            s["pairwise"].grad = None
            graphs.append(g)

    def step(i):
        if graphs:
            graphs[i % nsets].replay()
            fg.all_reduce()
            ops.COUNTERS["launches"] += launches_per_step
        else:
            eager_step(i)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled (20 ms period) from before the warm-up to the end of the timed region: same load throughout; the warm-up
    # runs for at least 0.5 s so that nvidia-smi is up and several samples land under load
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    warm_up(torch, dist, world, dev, step, max(args.warmup, 3))
    barrier()
    ops.COUNTERS["launches"] = 0
    ms = _timed(torch, dist, world, dev, step, args.steps, barrier)
    launches = ops.COUNTERS["launches"]
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                      # before the e2e arm and the profiled step overwrite the gradients
        last = dict(results[(args.steps - 1) % nsets])
        rows, urows = sample_rows(torch, B * N_POINTS, 32768, dev), sample_rows(torch, B * (N_POINTS // RATIO), 8192, dev)
        for name, r in (("out", rows), ("grad_pairwise", rows), ("grad_unary", urows)):
            last[name] = last[name].reshape(-1, last[name].shape[-1])[r]
        last["grad_params"] = torch.cat([g.reshape(-1) for g in last["grad_params"]])
        dump_outputs(args.dump_outputs, {**last, "out_rows": rows, "grad_unary_rows": urows})
    ms_step = ms / args.steps
    value = world * B * N_POINTS / (ms_step * 1e-3)

    # ---- e2e: host (pinned) inputs, H2D every step, D2H of the loss
    host = [{k: v.detach().cpu().pin_memory() for k, v in s.items() if k != "pos"} for s in sets[:2]]
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    loss_host = torch.zeros(1).pin_memory()

    # Two device-side staging buffers: the H2D copy of step i+1 runs on a copy stream while step i computes (the inputs of
    # every step still cross PCIe inside the timed region); fwd+bwd of each buffer is a captured CUDA graph when --graph.
    copy_stream = torch.cuda.Stream()
    # The int64 indices of the reference format are narrowed on the host (16 bits: every index < 65,536), copied packed and widened
    # on the device by the package's HostStager (crfconv_b200/host_io.py) — packing runs inside the timed region, every step.
    from crfconv_b200.host_io import HostStager
    limits = {"neighbor_idx": N_POINTS, "up_idx": N_POINTS // RATIO}
    # packing threads: this rank's share of the cores minus the main thread (which spins in cudaStreamSynchronize) and NCCL's
    cores_per_rank = len(os.sched_getaffinity(0)) // (1 if numa.get("cpus") else max(world, 1))
    pack_threads = args.pack_threads or max(1, min(16, cores_per_rank - 2))
    # both forms fill the SAME device tensors (the captured graphs read those): packed indices, or the int64 tensors as they are
    stagers_by_mode = {True: [HostStager(host[0], dev, index_limits=limits, threads=pack_threads, pack=True) for _ in range(2)]}
    stagers_by_mode[False] = [HostStager(host[0], dev, pack=False, dev_tensors=stagers_by_mode[True][j].dev) for j in range(2)]
    use_pack = args.pack_index != "off"
    stagers = stagers_by_mode[use_pack]
    stage = [st_.dev for st_ in stagers]
    h2d_ref_format = h2d
    for st_ in stage:
        st_["unary"].requires_grad_(True)
        st_["pairwise"].requires_grad_(True)
    ready = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    loss_dev = [torch.zeros(1, device=dev) for _ in range(2)]

    def fwd_bwd(j):
        st_ = stage[j]
        fg.zero()
        out = layer(st_["unary"], st_["pairwise"], st_["up_idx"], st_["neighbor_idx"])
        out.backward(cot)
        loss_dev[j].copy_(out.detach().sum().reshape(1))
        st_["unary"].grad = None
        st_["pairwise"].grad = None

    e2e_graphs = []
    if args.graph:
        for j in range(2):
            stagers[j].upload(host[j])
            torch.cuda.synchronize()
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                fwd_bwd(j)
            e2e_graphs.append(gph)

    # Index packing of step i+2 runs on a helper thread while step i computes and step i+1 copies: the main thread only enqueues.
    from concurrent.futures import ThreadPoolExecutor
    packer = ThreadPoolExecutor(1)
    packed = {}

    def prepare(i):
        packed[i] = packer.submit(stagers[i % 2].prepare, host[i % 2])

    def upload(i):
        j = i % 2
        packed.pop(i).result()
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done[j])                     # the previous user of this staging buffer has finished
            stagers[j].upload(host[j], copy_stream, prepared=True, defer_unpack=True)
            ready[j].record(copy_stream)

    def e2e_run(n):
        cur = torch.cuda.current_stream()
        for j in range(2):
            done[j].record(cur)
        prepare(0)
        upload(0)
        if n > 1:
            prepare(1)
        for i in range(n):
            j = i % 2
            cur.wait_event(ready[j])
            stagers[j].unpack(cur)                              # index widening: first kernels of the step, on the compute stream
            if e2e_graphs:
                e2e_graphs[j].replay()
            else:
                fwd_bwd(j)
            fg.all_reduce()
            loss_host.copy_(loss_dev[j], non_blocking=True)
            done[j].record(cur)
            if i + 1 < n:
                upload(i + 1)
            if i + 2 < n:
                prepare(i + 2)                                  # waits (on the helper thread) until step i's copies have left the pinned buffers
            cur.synchronize()                                   # the caller reads the loss on the host every step

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def e2e_timed(n):
        barrier()
        e0.record()
        e2e_run(n)
        e1.record()
        barrier()
        ms_ = e0.elapsed_time(e1)
        if world > 1:
            t_ = torch.tensor([ms_], device=dev)
            dist.all_reduce(t_, op=dist.ReduceOp.MAX)
            ms_ = float(t_.item())
        return ms_

    # --pack-index auto: whether narrowing the indices pays depends on the host (its packing threads compete with the other ranks'
    # packing and with the DMA reads for host memory bandwidth): both forms are timed for a few steps after their own warm-up and
    # the faster one — the same on every rank, the times are all-reduced — runs the timed region.
    tune = None
    if args.pack_index == "auto":
        trial = {}
        for mode in (True, False):
            stagers = stagers_by_mode[mode]
            e2e_run(3)
            trial[mode] = e2e_timed(8) / 8
        use_pack = trial[True] <= trial[False]
        tune = {"packed_ms_per_step": round(trial[True], 4), "plain_ms_per_step": round(trial[False], 4), "steps_each": 8}
    stagers = stagers_by_mode[use_pack]
    h2d = stagers[0].h2d_bytes(host[0])
    e2e_run(3)
    ms_e2e = e2e_timed(args.steps)
    e2e_value = world * B * N_POINTS / (ms_e2e / args.steps * 1e-3)
    probe = h2d_probe(torch, dev, host[0], barrier)              # every rank copies at once, no compute: the host-side ceiling
    if world > 1:
        t = torch.tensor([probe], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        probe = float(t.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel instrumented pass (CUDA events around every C-ABI launch on the launching stream)
    peaks, peak_src = measured_peaks()
    prof = ops.profile_calls(lambda: eager_step(0, reduce=False), repeats=3)    # rank 0 only: no collectives from here on
    total_k = sum(v["ms"] for v in prof.values())
    top = max(prof.items(), key=lambda kv: kv[1]["ms"])
    kernels = {k: {"kernel": _single_kernel_name(k), "ms_per_step": round(v["ms"], 4), "calls_per_step": v["calls"], "share": round(v["ms"] / total_k, 4),
                   "algo_bytes_per_step": v["bytes"], "achieved_gbs": round(v["bytes"] / (v["ms"] * 1e-3) / 1e9, 1) if v["ms"] > 0 else None}
               for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])}
    top_ach = top[1]["bytes"] / (top[1]["ms"] * 1e-3) / 1e9
    step_ach = ALGO_BYTES_PER_CLOUD * B / (ms_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(step_ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(step_ach / peaks["hbm_gbs"], 4), "frac_of_nominal_8TBs": round(step_ach / 8000.0, 4),
                "traffic": _ncu_traffic("step_dram_bytes"), "peak_source": peak_src,
                "scope": f"whole layer step (fwd+bwd, {launches_per_step or '?'} kernels in one CUDA graph): SURVEY.md §8(d) algorithmic bytes "
                         f"{ALGO_BYTES_PER_CLOUD} B per cloud x {B} clouds / CUDA-event step time",
                "algo_bytes_per_cloud": ALGO_BYTES_PER_CLOUD,
                "dominant_kernel": {"kernel": _single_kernel_name(top[0]), "call": top[0], "share_of_step": round(top[1]["ms"] / total_k, 4),
                                    "achieved": round(top_ach, 1), "frac": round(top_ach / peaks["hbm_gbs"], 4), "unit": "GB/s",
                                    "algo_bytes_per_launch": top[1]["bytes"] / max(top[1]["calls"], 1),
                                    "traffic": _ncu_traffic(top[0]),
                                    "note": "this kernel's own algorithmic bytes / its CUDA-event time in an eager instrumented pass"}}

    # ---- secondary metric of BASELINE.json: kNN queries/s (device-resident) on the same clouds
    pos = sets[0]["pos"]
    for _ in range(3):
        nn_.knn_batch(pos, pos, K_NBR)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(10):
        nn_.knn_batch(pos, pos, K_NBR)
    e1.record()
    torch.cuda.synchronize()
    knn_qps = 10 * B * N_POINTS / (e0.elapsed_time(e1) * 1e-3)

    _, _, cb = cpu_layer_points_per_s(clouds=B, repeats=4, warm=1)
    line = {"metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"single ContinuousGaussianCRFConv(128,64,64,steps=1) fwd+bwd, N=40960, Nc=10240, K=16, "
                                   f"{B} clouds per GPU per step (SURVEY.md §8 S1 / BASELINE configs[0] shape on the GPU)",
                       "config": "S1", "clouds_per_gpu": B, "precision": "3xTF32 tensor-core contractions, fp32 elsewhere" if ops.PRECISION == 0 else "TF32",
                       "launch": "one CUDA graph per input set, replayed" if args.graph else "eager (per-kernel launches from Python)",
                       "l2": f"rotating {nsets} input sets of {in_bytes / 2**20:.0f} MiB each (> {L2_BYTES / 2**20:.0f} MiB L2)",
                       "parallelism": f"dp{world}: clouds sharded, one NCCL all-reduce (AVG) of the flat gradient" if world > 1 else "single GPU"},
            "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps, "h2d_gbs_per_gpu": round(h2d / (ms_e2e / args.steps * 1e-3) / 1e9, 2),
                    "h2d_probe_gbs_per_gpu": round(probe, 2), "numa": numa,
                    "h2d_bytes_reference_format": h2d_ref_format,
                    "index_packing": {"mode": args.pack_index, "used": bool(use_pack), "auto_tune": tune,
                                      "how": ("int64 indices narrowed to 16 bits on the host (helper thread + %d packing threads, range-checked, "
                                              "every step, inside the timed region), widened on the device" % pack_threads) if use_pack
                                             else "int64 index tensors copied as they are"}},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "kernels": kernels,
            "knn": {"metric": "kNN queries/s", "value": knn_qps, "unit": "queries/s", "config": f"B={B}, N=Q=40960, K=16, device-resident"},
            "cpu_baseline": cb}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_gpu_network(args, rank, local_rank, world, dev, numa):
    """--config C3 / C4 / C5: the whole PointConvResNet fwd + cross-entropy + bwd."""
    import torch
    import torch.distributed as dist
    import torch.nn.functional as Fn
    from crfconv_b200 import losses, ops, train_dp
    from crfconv_b200.distributed import FlatGradients
    from crfconv_b200.graphs import GraphedStep
    from crfconv_b200.point_conv_big import PointConvResNet
    cfg = NET_CONFIGS[args.config]
    B, N, ncls = args.clouds or cfg["clouds"], cfg["points"], cfg["classes"]
    torch.manual_seed(1234)
    net = PointConvResNet(6, ncls).to(dev).train()
    grads = FlatGradients(net, direct=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    pos, feat, lab, gen = train_dp.synthetic_shard(B, N, ncls, dev, seed=77 + rank)
    data = train_dp.make_batch(pos, feat, lab, generator=gen)
    target = (lab.reshape(-1) - 1).contiguous()

    def net_step():
        grads.zero()
        loss = losses.cross_entropy(net(data), target)        # the package's criterion kernels (csrc/loss.cu)
        loss.backward()
        return loss.detach()

    ops.COUNTERS["launches"] = 0
    gs = GraphedStep(net_step) if args.graph else None
    launches_per_step = 0

    last = {}

    def step(i):
        if gs is not None:
            last["loss"] = gs.replay()
        else:
            last["loss"] = net_step()
        if world > 1:
            grads.all_reduce()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    warm_up(torch, dist, world, dev, step, max(args.warmup, 3), chunk=4)
    barrier()
    # the classifier's dropout draws a new mask every step and the warm-up ends on a clock: reseeding here gives the timed steps
    # the same masks in every run
    torch.cuda.manual_seed(1234)
    ms = _timed(torch, dist, world, dev, step, args.steps, barrier)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                      # before the eager step below overwrites the gradients
        dump_outputs(args.dump_outputs, {"loss": last["loss"].reshape(1), "grad_params": grads.flat[:grads.numel]})
    ms_step = ms / args.steps
    value = world * B * N / (ms_step * 1e-3)
    ops.COUNTERS["launches"] = 0
    net_step()                                                           # one eager step: counts this package's kernel launches
    launches_per_step = ops.COUNTERS["launches"]
    torch.cuda.synchronize()

    # ---- e2e: points, features and labels come from pinned host memory every step; the pyramid (10 kNN calls + subsampling) is
    # built on the GPU inside the timed region; the loss is read back on the host
    hp, hf, hl = pos.cpu().pin_memory(), feat.cpu().pin_memory(), lab.cpu().pin_memory()
    h2d = sum(t.numel() * t.element_size() for t in (hp, hf, hl))
    loss_host = torch.zeros(1).pin_memory()

    def e2e_step(i):
        p, f, l = hp.to(dev, non_blocking=True), hf.to(dev, non_blocking=True), hl.to(dev, non_blocking=True)
        d = train_dp.make_batch(p, f, l, generator=gen)               # the pyramid: 10 kNN calls + subsampling, on the GPU, eager
        if gs is not None:
            # batches have static shapes: the new pyramid is copied INTO the captured step's input tensors and the graph is replayed
            GraphedStep.copy_inputs(data, d)
            target.copy_(l.reshape(-1) - 1, non_blocking=True)
            loss = gs.replay()
        else:
            grads.zero()
            loss = losses.cross_entropy(net(d), l.reshape(-1) - 1)
            loss.backward()
        if world > 1:
            grads.all_reduce()
        loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for i in range(2):
        e2e_step(i)
    n_e2e = args.steps
    ms_e2e = _timed(torch, dist, world, dev, e2e_step, n_e2e, barrier)
    e2e_value = world * B * N / (ms_e2e / n_e2e * 1e-3)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks, peak_src = measured_peaks()
    A = network_algo_bytes(N, ncls)
    ach = A * B / (ms_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(ach / peaks["hbm_gbs"], 4),
                "traffic": _ncu_traffic(f"{args.config}_step_dram_bytes"), "peak_source": peak_src, "algo_bytes_per_cloud": A,
                "scope": "whole network step: shape walker over 10 ResNetBBlocks + 4 CRF layers + classifier with SURVEY.md §8(d)'s formulas"}
    _, _, cb = cpu_network_points_per_s(cfg, clouds=2, repeats=2, warm=1)
    line = {"metric": "PointConvResNet fwd+bwd points/s", "value": value, "unit": "points/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"PointConvResNet(6,{ncls},use_crf=True,steps=1) fwd + cross-entropy + bwd, {cfg['name']}; {B} clouds per GPU per step, "
                                   "5-level kNN pyramid (K=16, ratios 4/4/4/4/2) prebuilt on the device for `value`, rebuilt every step for `e2e`",
                       "config": args.config, "clouds_per_gpu": B, "points": N, "classes": ncls,
                       "launch": "one CUDA graph, replayed" if args.graph else "eager",
                       "l2": f"working set of a step ({A * B / 2**20:.0f} MiB algorithmic) exceeds the {L2_BYTES / 2**20:.0f} MiB L2",
                       "parallelism": f"dp{world}: clouds sharded, one NCCL all-reduce (AVG) of the flat gradient" if world > 1 else "single GPU"},
            "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / n_e2e,
                    "steps": n_e2e, "numa": numa, "note": ("pyramid built eagerly on the GPU every step, copied into the captured step's inputs, network step replayed as one CUDA graph"
                             if args.graph else "eager launches")},
            "gpu_launches": launches_per_step * args.steps, "clocks": clocks, "roofline": roofline, "cpu_baseline": cb}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100, help="timed steps (--impl reference runs this many CPU passes: keep it small there)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="S1", choices=["S1", "C3", "C4", "C5"])
    ap.add_argument("--clouds", type=int, default=0, help="clouds per GPU per step (default: 6 for S1/C3, 8 for C4, 2 for C5)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pack-index", default="auto", choices=["auto", "on", "off"],
                    help="e2e arm: narrow the int64 index tensors to 16 bits on the host before the copy (auto: time both forms, keep the faster)")
    ap.add_argument("--pack-threads", type=int, default=0, help="host threads of the index packing (default: min(16, cores per rank - 2); measured 1 / 2 / 4 / 8 / 16 threads: 2.84 / 2.18 / 2.04 / 2.05 / 1.92 ms per step)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="launch every kernel from Python instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned as DIR/<name>.npy (float32; S1: a fixed sample of the rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-launch under torch.distributed.run, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 2000), os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--config", args.config, "--clouds", str(args.clouds), "--pack-index", args.pack_index,
               "--pack-threads", str(args.pack_threads)] + ([] if args.graph else ["--no-graph"]) \
            + (["--dump-outputs", args.dump_outputs] if args.dump_outputs else [])
        sys.exit(subprocess.call(cmd))
    run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
