#!/usr/bin/env python
"""Benchmark of the SPARF ray-marching hot path (BASELINE.json metric: rays/s, fwd+bwd, 128 samples/ray).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c2h|c3|c4|c5] [--impl ours|reference]
                    [--engine auto|simt_fp32|tc_3x|tc_3x_w1 (reduced precision, labelled so)] [--graph 0|1] [--device cpu|cuda (reference arm)]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic ray batch of a BASELINE config, through the public API
(`Graph.render_image_at_specific_rays` + the loss module's `compute_loss` + `backward()`), gradients zeroed each step:

    c1   BASELINE config 1 (the reference's own CPU-runnable case): one 32x32 view, identity pose, 256 rays x 64 samples
    c2   (default; the driver's line) DTU-shaped 3 views 300x400, fixed GT poses, 3 x 341 = 1023 rays x 128 coarse
         samples, photometric loss -- the "1024-ray / 128-sample" headline shape
    c2h  the real DTU setting of config 2: + hierarchical fine pass (128 resampled + 128 coarse = 256 through nerf_fine)
    c3   c2h + BARF coarse-to-fine mask + SE(3) pose refinement (9-D pose embedding, gradients to the poses)
    c4   LLFF-shaped 3 views 378x504, 3 x 682 = 2046 rays x 128 samples of inverse depth, joint poses, full SPARF step:
         photometric + multi-view correspondence + depth-consistency losses (6 render calls)
    c5   Replica-shaped 9 views 340x600, 9 x 455 = 4095 rays, hierarchical, pose gradients; STRONG scaling: the batch
         is sharded over the N GPUs, one NCCL all-reduce of [d theta_c | d theta_f | d xi] per step

Timing: W warm-up steps, then K steps between a barrier + synchronize on both sides; every step is bracketed by its own
CUDA events on the launching stream, with an L2 flush (256 MiB memset) between steps outside the event pairs and (default)
a synchronize after each step; ms_per_step = mean of the K intervals, MAX over ranks.  `--sync-each-step 0` enqueues the K
steps back to back instead.  Clocks / throttle reasons are sampled with nvidia-smi during the timed region.  Prints ONE JSON line (rank 0).

`--impl reference` times the torch restatement of the reference's hot path (oracle/sparf_oracle.py, pinned to the
reference by tests/golden; config c2) on the host cores (`--device cuda`: on the GPU, the torch/cuBLAS path SURVEY 8d
calls "the kernel to beat").  The N = 1 line of our arm carries both as `cpu_baseline` and `torch_gpu_baseline`.

`--dump-outputs DIR` writes what the last timed step of our arm computed, as DIR/<name>.npy: the loss, every parameter
gradient (`grad.graph.*`, `grad.pose.*`) and the tensors the render call returned (`render.*`), rank 0.  The inputs
(scene, weights, ray draws, sampling noise) are seeded, so two builds run with the same arguments can be compared
array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

# algorithmic work (SURVEY.md 8d): MACs per MLP sample-evaluation; forward = 2 MACs, forward + backward = 6 MACs
MACS_PER_SAMPLE = 63 * 256 + 3 * 256 * 256 + 319 * 256 + 2 * 256 * 256 + 256 * 257 + 283 * 128 + 128 * 3  # 527 872

CONFIGS = {
    "c1": dict(B=1, H=32, W=32, focal=32.0, rand_rays=256, S=64, fine=False, S_fine=64, depth_range=(0.5, 2.5),
               depth_param="metric", poses=False, c2f=None, progress=None, loss_type="photometric", scaling="weak",
               identity=True,
               desc="BASELINE config 1: single 32x32 synthetic view, identity pose, 256 rays x 64 coarse samples, photometric loss, fwd+bwd (the reference's CPU-runnable case)"),
    "c2": dict(B=3, H=300, W=400, focal=400.0, rand_rays=1024, S=128, fine=False, S_fine=128, depth_range=(1.2, 5.2),
               depth_param="metric", poses=False, c2f=None, progress=None, loss_type="photometric", scaling="weak",
               desc="DTU-shaped 3 views 300x400, fixed GT poses, 3x341=1023 rays x 128 coarse samples, photometric loss, fwd+bwd"),
    "c2h": dict(B=3, H=300, W=400, focal=400.0, rand_rays=1024, S=128, fine=True, S_fine=128, depth_range=(1.2, 5.2),
                depth_param="metric", poses=False, c2f=None, progress=None, loss_type="photometric", scaling="weak",
                desc="DTU-shaped 3 views 300x400, fixed GT poses, 1023 rays, hierarchical 128 coarse + 256 fine-network samples, photometric loss (coarse + fine), fwd+bwd"),
    "c3": dict(B=3, H=300, W=400, focal=400.0, rand_rays=1024, S=128, fine=True, S_fine=128, depth_range=(1.2, 5.2),
               depth_param="metric", poses=True, c2f=(0.1, 0.5), progress=0.3, loss_type="photometric", scaling="weak",
               desc="DTU-shaped joint pose-NeRF (BARF c2f mask + 9-D pose embeddings with gradients), 1023 rays, hierarchical 128 + 256 samples, photometric loss, fwd+bwd"),
    "c4": dict(B=3, H=378, W=504, focal=500.0, rand_rays=2048, S=128, fine=False, S_fine=128, depth_range=(1, 0),
               data_depth_range=(0.5, 8.0), depth_param="inverse", poses=True, c2f=(0.4, 0.7), progress=0.55,
               loss_type="photometric_and_corres_and_depth_cons", scaling="weak",
               desc="LLFF-shaped 3 views 378x504, joint poses, 3x682=2046 rays x 128 inverse-depth samples, full SPARF step: photometric + correspondence + depth-consistency (6 render calls), fwd+bwd"),
    "c5": dict(B=9, H=340, W=600, focal=600.0, rand_rays=4096, S=128, fine=True, S_fine=128, depth_range=(0.1, 4.5),
               depth_param="metric", poses=True, c2f=(0.4, 0.7), progress=0.55, loss_type="photometric", scaling="strong",
               desc="Replica-shaped 9 views 340x600, 9x455=4095 rays sharded over the GPUs, hierarchical 128 + 256 samples, pose gradients in the reduced buffer, photometric loss, fwd+bwd"),
}
METRIC = "rays/sec (fwd+bwd, 128 samples/ray)"
DTYPE = ("fp32 in / out; GEMMs on tcgen05 kind::f16 with a 3-pass error-compensated split (fp16 halves forward, bf16 "
         "halves backward), fp32 TMEM accumulation; fp32 CUDA cores for encoding / activations / compositing")
ENGINE_DTYPE = {"auto": DTYPE, "tc_3x": DTYPE,
                "tc_3x_w1": "REDUCED PRECISION (non-default engine, not a parity number): as tc_3x, but the weight gradients in "
                            "ONE bf16 pass over the hi halves of the saved images",
                "tc_1x": "REDUCED PRECISION (non-default engine, not a parity number): single 16-bit pass forward"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"),
                    hbm_gbs=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self, wait_s=5.0):
        """Launch `nvidia-smi -lms 50` and block until its first row arrives (it needs ~0.5 s to come up; the timed
        region of a short run would otherwise be over before the first sample)."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < wait_s:
                time.sleep(0.02)
            self.rows.clear()   # samples from here on fall inside the measured regions
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=smax, reasons=sorted(reasons),
                    samples=len(sm))


# ------------------------------------------------------------------------------------------------ workload
class _TrainData:
    def __init__(self, d, n):
        self.all, self.n = d, n

    def __len__(self):
        return self.n


def build_problem(cfg_name, device, seed=0, stratified=True):
    """Model + data + loss module of one BASELINE config on our path.  Returns a namespace with `.forward_backward(ray_idx)`."""
    import common
    cfg = CONFIGS[cfg_name]
    B, H, W = cfg["B"], cfg["H"], cfg["W"]
    opt = common.make_opt(S=cfg["S"], S_fine=cfg["S_fine"], fine=cfg["fine"], depth_param=cfg["depth_param"],
                          depth_range=cfg["depth_range"], rand_rays=cfg["rand_rays"], stratified=stratified, noise=False,
                          barf_c2f=cfg["c2f"])
    opt.loss_type = cfg["loss_type"]
    if "corres" in cfg["loss_type"]:
        opt.loss_weight.corres = -3.0
        opt.loss_weight.depth_cons = -3.0
    torch.manual_seed(seed)
    np.random.seed(seed)
    data = common.make_scene(seed, B, H, W, focal=cfg["focal"], identity=cfg.get("identity", False))
    data.depth_range = torch.tensor([list(map(float, cfg.get("data_depth_range", cfg["depth_range"])))] * B)
    for k in ("image", "intr", "pose", "depth_range", "idx"):
        data[k] = data[k].to(device)
    sd = common.det_weights(opt, seed, progress=cfg["progress"])
    sd_fine = common.det_weights(opt, seed + 77, progress=cfg["progress"]) if cfg["fine"] else None
    from sparf_b200.losses import define_loss
    from sparf_b200.poses_models import FirstTwoColunmnsPoseParameters
    from sparf_b200.renderer import Graph
    pose_net = None
    if cfg["poses"]:
        init = common.perturb_poses(data.pose.cpu(), seed, sigma=0.02).to(device)
        pose_net = FirstTwoColunmnsPoseParameters(opt, nbr_poses=B, initial_poses_w2c=init, device=device).to(device)

        class PoseGraph(Graph):   # joint_pose_nerf_trainer.py:710-722, train mode
            def get_w2c_pose(self, opt, data_dict, mode=None):
                return pose_net.get_w2c_poses()

        net = PoseGraph(opt, device)
    else:
        net = Graph(opt, device)
    net.nerf.load_state_dict(sd)
    if cfg["fine"]:
        net.nerf_fine.load_state_dict(sd_fine)
    net.to(device).train()
    flow = common.FakeFlowNet(B, H, W) if "corres" in cfg["loss_type"] else None
    # sync-free fixed-shape mode of the SPARF losses (SURVEY 8f.2): the step is one CUDA graph
    loss_module = define_loss(opt.loss_type, opt, net, _TrainData(data, B), device, flow_net=flow, device_side=True)
    modules = [net] + ([pose_net] if pose_net is not None else [])
    pr = argparse.Namespace(cfg=cfg, opt=opt, data=data, net=net, pose_net=pose_net, loss_module=loss_module,
                            modules=modules, iteration=10)

    needs_poses = "corres" in cfg["loss_type"] or "depth_cons" in cfg["loss_type"]

    def forward_backward(ray_idx):
        data["iter"] = pr.iteration
        out = net.render_image_at_specific_rays(opt, data, iter=pr.iteration, ray_idx=ray_idx, mode="train")
        if needs_poses:     # nerf_trainer.py:239-240: the current pose estimates, with their autograd history
            data.poses_w2c = net.get_w2c_pose(opt, data, mode="train")
        loss = loss_module.compute_loss(opt, data, out, iteration=pr.iteration, mode="train")[0]["all"]
        loss.backward()
        if needs_poses:     # do not keep the step's autograd graph alive into the next step (or a graph capture)
            data.pop("poses_w2c", None)
        return loss.detach(), {k: v.detach() for k, v in out.items() if torch.is_tensor(v)}

    pr.forward_backward = forward_backward
    return pr


def rays_per_view(cfg, rank=0, world=1):
    n = cfg["rand_rays"] // cfg["B"]
    if cfg["scaling"] == "strong" and world > 1:
        from sparf_b200.distributed import shard_range
        lo, hi = shard_range(n, rank, world)
        return hi - lo
    return n


def quiet_nccl_banner():
    """NCCL_DEBUG=VERSION (set on some boxes) makes NCCL print "NCCL version ..." on STDOUT, in front of the one JSON line
    this script owes its caller; keep stdout clean (an explicit INFO / TRACE request is left alone)."""
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        del os.environ["NCCL_DEBUG"]       # (WARN would still print the banner: every level >= VERSION does)


def run_ours(args):
    quiet_nccl_banner()
    import sparf_b200
    from sparf_b200 import _lib, ops
    from sparf_b200.distributed import FlatGradients, shard_range
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    sparf_b200.set_engine(args.engine)
    L = _lib.lib()
    cfg = CONFIGS[args.config]
    strong = cfg["scaling"] == "strong"
    # weak scaling: every rank its own scene-independent batch (seed = rank); strong: one global batch, sharded
    pr = build_problem(args.config, dev, seed=0 if strong else rank)
    pr.net.device_side_rng = True
    pr.loss_module.check_finite = False      # no host synchronisation inside the step (see sparf_b200/losses.py)
    if world > 1:   # identical replicas of the MLPs / poses on every rank
        for m in pr.modules:
            for p in m.parameters():
                dist.broadcast(p.data, 0)
    fg = FlatGradients(pr.modules)            # [d theta_coarse | d theta_fine | d pose]: one buffer, one all-reduce
    flat = fg.flat
    HW = cfg["H"] * cfg["W"]
    n_view_global = cfg["rand_rays"] // cfg["B"]
    n_view = rays_per_view(cfg, rank, world)
    g = torch.Generator(device="cpu").manual_seed(1234 + (0 if strong else rank))
    n_total = args.warmup + args.steps

    def draw():
        idx = torch.randperm(HW, generator=g)[:n_view_global]
        if strong and world > 1:
            lo, hi = shard_range(n_view_global, rank, world)
            idx = idx[lo:hi]
        return idx.pin_memory()

    idx_host = [draw() for _ in range(2 * n_total + 1)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    loss_host = torch.zeros((), pin_memory=True)
    scale = (n_view / n_view_global) if (strong and world > 1) else 1.0   # local mean -> share of the global mean

    def local_step(ray_idx_dev):   # everything of a step except the cross-rank exchange -> (loss, render outputs)
        flat.zero_()
        out = pr.forward_backward(ray_idx_dev)
        if scale != 1.0:
            flat.mul_(scale)
        return out

    def step(ray_idx_dev):
        out = local_step(ray_idx_dev)
        if world > 1:
            dist.all_reduce(flat)  # one NCCL all-reduce of [d theta | d xi] per step (SURVEY 8e)
        return out

    graphed, ar_in_graph, launches_per_graph = None, False, None
    evals_per_step = None
    ops.EVALS["fwd"] = ops.EVALS["bwd"] = 0
    step(idx_host[-1].to(dev))     # one eager step: lazy initialisation + the per-step evaluation counts
    torch.cuda.synchronize()
    evals_per_step = dict(ops.EVALS)
    if args.graph and cfg.get("graph", True):
        from sparf_b200.graphs import GraphedStep
        static_idx = idx_host[0].to(dev)
        c0 = L.sparf_launch_count()
        try:
            if world > 1 and args.allreduce_in_graph:
                graphed = GraphedStep(step, (static_idx,), warmup=2)      # NCCL all-reduce captured with the step
                ar_in_graph = True
            else:
                graphed = GraphedStep(local_step, (static_idx,), warmup=2)
            launches_per_graph = (L.sparf_launch_count() - c0) // 3   # 2 eager warm-ups + the capture
        except Exception as e:   # e.g. a config whose losses still take host decisions: run it eagerly
            if world > 1 and args.allreduce_in_graph:
                raise
            sys.stderr.write("bench: CUDA-graph capture of config %s failed (%s: %s); running eagerly\n"
                             % (args.config, type(e).__name__, str(e)[:200]))
            graphed = None
            torch.cuda.synchronize()

    def graph_step(ray_idx_src):
        out = graphed(ray_idx_src)
        if world > 1 and not ar_in_graph:
            dist.all_reduce(flat)
        return out

    def timed(n_warm, n_steps, e2e, use_graph=False):
        # every step is bracketed by its own pair of CUDA events on the launching stream with the L2 flush outside the
        # pair; barrier + synchronize on both sides of the whole loop.  By default the host also synchronises after each
        # step (--sync-each-step 0: the steps are enqueued back to back; measured 1.364 vs 1.350 ms on the same
        # power-capped box, the launch latency of a graph replay on an idle device is below the noise).  The
        # end-to-end arm always waits for every step's loss on the host (a caller that reads its result).
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        events, render = [], None
        for i in range(n_warm + n_steps):
            src = idx_host[(n_total if e2e else 0) + i]
            if not e2e:
                ray_idx_dev = src.to(dev, non_blocking=True)
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if e2e:  # host buffers in, host scalar out, inside the timed region
                ray_idx_dev = src if use_graph else src.to(dev, non_blocking=True)
            loss, render = graph_step(ray_idx_dev) if use_graph else step(ray_idx_dev)
            if e2e:
                loss_host.copy_(loss.detach(), non_blocking=True)
            e1.record()
            if e2e or args.sync_each_step:
                torch.cuda.synchronize()
            events.append((e0, e1))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        times = [a.elapsed_time(b) for a, b in events[n_warm:]]
        t = torch.tensor([sum(times)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), times, render

    rays_local = cfg["B"] * n_view
    rays_per_step = cfg["B"] * n_view_global if strong else rays_local * world
    ops.PROFILE.clear()
    timed(args.warmup, 0, False)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = L.sparf_launch_count()
    ops.PROFILE.clear()
    ops.PROFILE_ON[0] = True
    total_ms, times, _ = timed(0, args.steps, False)
    ops.PROFILE_ON[0] = False
    launches = L.sparf_launch_count() - launches0
    mlp_ms = ops.profile_total_ms()   # MLP kernel groups timed with CUDA events in the eager pass (same kernels)
    eager_ms_per_step = total_ms / args.steps
    if graphed is not None:           # the reported step: one CUDA-graph replay per step
        timed(args.warmup, 0, False, use_graph=True)
        total_ms, times, _ = timed(0, args.steps, False, use_graph=True)
        launches = launches_per_graph * args.steps
    e2e_ms, _, render = timed(args.warmup, args.steps, True, use_graph=graphed is not None)
    if args.dump_outputs and rank == 0:    # before the all-reduce timing below, which keeps summing into the gradients
        arrays = {"loss": loss_host}
        for prefix, m in (("grad.graph", pr.net), ("grad.pose", pr.pose_net)):
            for name, p in (m.named_parameters() if m is not None else ()):
                if p.grad is not None:
                    arrays["%s.%s" % (prefix, name)] = p.grad
        arrays.update(("render." + k, v) for k, v in render.items() if v.is_floating_point())
        dump_outputs(args.dump_outputs, arrays)
    # cost of the collective alone (rank 0's view): the all-reduce of the flat buffer, timed back to back
    ar_us = None
    if world > 1:
        for _ in range(5):
            dist.all_reduce(flat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        e0.record()
        for _ in range(20):
            dist.all_reduce(flat)
        e1.record()
        torch.cuda.synchronize()
        ar_us = e0.elapsed_time(e1) * 1e3 / 20
    clocks = sampler.stop() if rank == 0 else None   # sampled over the device-timed AND the end-to-end region
    launched_as_graph = graphed is not None
    if world > 1:
        # a CUDA graph that captured NCCL kernels must be gone before the communicator is torn down
        graphed = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
    if rank != 0:
        shutdown_distributed(dist)
        return
    peaks = load_peaks()
    ms_per_step = total_ms / args.steps
    value = rays_per_step / (ms_per_step * 1e-3)
    # algorithmic FLOP of this rank's step: every MLP sample-evaluation the step issued (forward 2 MACs, backward 4 MACs)
    flop_step_gpu = (2 * evals_per_step["fwd"] + 4 * evals_per_step["bwd"]) * MACS_PER_SAMPLE
    mlp_ms_per_step = mlp_ms / args.steps if mlp_ms else None
    # MLP kernel group: CUDA events around sparf_mlp_forward* / sparf_mlp_backward* in the eager pass.  The graph replay
    # runs the same kernels with smaller gaps, so when a whole replayed step is shorter than the eager MLP group, the
    # step time is the (conservative) upper bound of the group's duration.
    group_ms = min(mlp_ms_per_step, ms_per_step) if mlp_ms_per_step else ms_per_step
    achieved = flop_step_gpu / (group_ms * 1e-3) / 1e12
    roofline = dict(bound="tensor", kernel="MLP fwd+bwd kernels of one step (sparf_mlp_forward_tape + sparf_mlp_backward_tape: "
                                           "tc_mlp_fwd / dgrad / wgrad + small kernels)",
                    achieved=achieved, peak=peaks["bf16_tflops"], unit="TFLOP/s", frac=achieved / peaks["bf16_tflops"],
                    peak_source=peaks["source"] + ", burst bf16",
                    frac_of_sustained=(achieved / peaks["bf16_tflops_sustained"]) if peaks["bf16_tflops_sustained"] else None,
                    three_pass_ceiling=1.0 / 3.0,
                    flop_per_launch_group=flop_step_gpu, ms_per_launch_group=group_ms,
                    ms_per_launch_group_eager_events=mlp_ms_per_step,
                    mlp_sample_evals_per_step=evals_per_step,
                    traffic=TRAFFIC.get((args.engine if args.engine != "auto" else "tc_3x", args.config)),
                    traffic_source=TRAFFIC_SOURCE.get(args.engine if args.engine != "auto" else "tc_3x"), engine=args.engine)
    cpu = tgb = None
    if world == 1 and not args.no_baselines:   # reported on rank 0 at N = 1 only
        graphed = None
        torch.cuda.empty_cache()
        try:
            tgb = torch_gpu_baseline(args.config, dev)
        except Exception as e:
            tgb = dict(unavailable="%s: %s" % (type(e).__name__, str(e)[:160]))
        try:
            cpu = cpu_baseline(args.config, budget_s=25.0)
        except RuntimeError as e:   # a config the oracle port does not cover
            cpu = dict(unavailable="%s: %s" % (type(e).__name__, str(e)[:160]))
    line = dict(metric=METRIC, value=value, unit="rays/s", n_gpus=world, steps=args.steps,
                warmup=args.warmup, ms_per_step=ms_per_step, higher_is_better=True, scaling=cfg["scaling"], vs_baseline=None,
                dtype=ENGINE_DTYPE.get(args.engine, "fp32 (CUDA cores)"), data="synthetic",
                config=dict(workload=cfg["desc"], name=args.config, rays_per_gpu=rays_local, global_rays=rays_per_step,
                            samples_per_ray=cfg["S"], fine_samples_per_ray=(cfg["S"] + cfg["S_fine"]) if cfg["fine"] else 0,
                            l2_flush_between_steps=True,
                            launch="one CUDA-graph replay per step" if launched_as_graph else "eager",
                            eager_ms_per_step=eager_ms_per_step,
                            timing="per-step CUDA-event intervals on the launching stream (L2 flush between steps outside the "
                                   "intervals, %s), barrier + synchronize on both sides; sum, max over ranks"
                                   % ("synchronize after every step" if args.sync_each_step else "steps enqueued back to back"),
                            parallelism="dp%d (ray sharding, one NCCL all-reduce of [MLP | pose] grads per step%s)"
                                        % (world, ", captured in the step's CUDA graph" if ar_in_graph else ""),
                            allreduce_us=ar_us, allreduce_bytes=int(flat.numel() * 4)),
                clocks=clocks,
                e2e=dict(value=rays_per_step / (e2e_ms / args.steps * 1e-3), unit="rays/s",
                         h2d_bytes_per_step=n_view * 8, d2h_bytes_per_step=4),
                gpu_launches=int(launches), roofline=roofline, cpu_baseline=cpu, torch_gpu_baseline=tgb)
    print(json.dumps(line), flush=True)
    if world > 1:
        shutdown_distributed(dist)


def dump_outputs(dirname, arrays, limit_bytes=64 << 20):
    """Write every tensor of `arrays` as dirname/<name>.npy in float32 (float64 stays float64).  If they come to more than
    `limit_bytes` together, each array above an equal share of the limit is cut to a fixed, seeded sample of its
    flattened values (the same positions on every run of the same configuration)."""
    os.makedirs(dirname, exist_ok=True)
    host = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    host = {k: v if v.dtype == np.float64 else v.astype(np.float32) for k, v in host.items()}
    share = limit_bytes // max(len(host), 1)
    big = sum(v.nbytes for v in host.values()) > limit_bytes
    for k, v in host.items():
        if big and v.nbytes > share:
            keep = np.sort(np.random.default_rng(0).choice(v.size, share // v.itemsize, replace=False))
            v = v.reshape(-1)[keep]
        np.save(os.path.join(dirname, k + ".npy"), v)


def shutdown_distributed(dist, grace_s=15.0):
    """destroy_process_group() with a watchdog: the measurement is printed already, a communicator that does not tear
    down cleanly must not keep the launcher (and the GPUs) busy until somebody's timeout fires."""
    done = threading.Event()

    def watchdog():
        if not done.wait(grace_s):
            sys.stderr.write("bench: destroy_process_group() did not return within %.0f s; exiting\n" % grace_s)
            sys.stderr.flush()
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()
    try:
        dist.destroy_process_group()
    finally:
        done.set()


# dram__bytes_read.sum + dram__bytes_write.sum of the MLP kernel group of one step, from `ncu --set full` captures
# (taped forward 1.228 GB, dgrad 1.138 GB, wgrad 2.391 GB at the c2 shape)
TRAFFIC = {("tc_3x", "c2"): 4.770e9, ("tc_3x_w1", "c2"): 2.582e9}
TRAFFIC_SOURCE = {"tc_3x": "profiles/r02_ncu_chain.md (ncu --set full of tc_mlp_fwd / dgrad / wgrad, per step)",
                  "tc_3x_w1": "profiles/r02_ncu_chain_w1.md (ncu --set full of tc_mlp_fwd / dgrad / wgrad, per step)"}


# ------------------------------------------------------------------------------------------------ reference arms
def reference_step_fn(cfg_name, device):
    """One step of the hot path through the oracle port of the reference (oracle/sparf_oracle.py, config c2 only) on
    `device`.  Returns (step, kind)."""
    cfg = CONFIGS[cfg_name]
    HW = cfg["H"] * cfg["W"]
    n_view = cfg["rand_rays"] // cfg["B"]
    g = torch.Generator().manual_seed(0)
    if cfg_name != "c2":
        raise RuntimeError("the oracle port only covers config c2")
    import common
    from oracle import sparf_oracle as O
    opt = common.make_opt(S=cfg["S"], fine=False, stratified=True)
    data = common.make_scene(0, cfg["B"], cfg["H"], cfg["W"], focal=cfg["focal"])
    sd = common.det_weights(opt, 0)
    to = lambda x: x.to(device)
    params = {k: to(v).clone().requires_grad_(k != "progress") for k, v in sd.items()}
    drange = to(torch.tensor(cfg["depth_range"]))
    pose, intr, image = to(data.pose), to(data.intr), to(data.image)

    def step():
        for p in params.values():
            p.grad = None
        ray_idx = to(torch.randperm(HW, generator=g)[:n_view])
        center, ray = O.rays_from_ray_idx(pose, intr, cfg["H"], cfg["W"], ray_idx)
        rand = to(torch.rand(cfg["B"], n_view, cfg["S"], 1, generator=g))
        out = O.render(opt, params, None, center, ray, drange, mode="train", rand=rand)
        loss = O.photometric_loss(out, image, ray_idx)
        loss.backward()
        return loss.detach()

    return step, "port"


def pick_cpu_threads(step):
    """torch CPU ops of this size do not scale to every core of a 100+ core host (the reference has the same
    behaviour): time one step at a few thread counts and keep the fastest."""
    cores = os.cpu_count() or 1
    best = (None, float("inf"))
    tried = {}
    # (all cores of a 100+ core host is never the optimum for this size -- measured 12.6 s/step at 128 threads vs 1.4 s
    #  at 16..32 -- and would eat the time budget of the CPU leg: stop at 64)
    cands = sorted({min(cores, 8), min(cores, 16), min(cores, 32), min(cores, 64)})
    torch.set_num_threads(min(cores, 32))
    step()                                   # warm-up (allocator, lazy initialisation)
    t0 = time.perf_counter()
    step()
    probe = time.perf_counter() - t0
    if probe > 4.0:                          # big configs: keep the CPU leg bounded, search two counts only
        cands = sorted({min(cores, 16), min(cores, 32)})
        tried[min(cores, 32)] = round(probe, 3)
        best = (min(cores, 32), probe)
        cands = [n for n in cands if n != min(cores, 32)]
    for n in cands:
        torch.set_num_threads(n)
        if probe <= 4.0:
            step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        tried[n] = round(dt, 3)
        if dt < best[1]:
            best = (n, dt)
    torch.set_num_threads(best[0])
    return best[0], tried


def cpu_baseline(cfg_name, budget_s=25.0):
    cfg = CONFIGS[cfg_name]
    cores = os.cpu_count() or 1
    step, kind = reference_step_fn(cfg_name, torch.device("cpu"))
    used, tried = pick_cpu_threads(step)
    n_rays = cfg["B"] * (cfg["rand_rays"] // cfg["B"])
    t0 = time.perf_counter()
    n = 0
    while n < 2 or (time.perf_counter() - t0 < budget_s and n < 50):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    return dict(value=n_rays / dt, unit="rays/s", cores=used, host_cores=cores, kind=kind,
                sample="%d full steps of config %s (%d rays) through %s on the host cores, torch CPU fp32, best thread "
                       "count of %s = %d, %.2f s/step"
                       % (n, cfg_name, n_rays, "oracle/sparf_oracle.py", tried, used, dt))


def torch_gpu_baseline(cfg_name, dev, steps=10, warmup=3):
    """The reference's own PyTorch path on THIS GPU (30 cuBLAS SGEMMs + ~100 ATen kernels per render call,
    frequency_nerf.py:162-170): fp32 with TF32 off (the reference's default arithmetic) and with TF32 on."""
    cfg = CONFIGS[cfg_name]
    n_rays = cfg["B"] * (cfg["rand_rays"] // cfg["B"])
    out = dict(unit="rays/s")
    step, kind = reference_step_fn(cfg_name, dev)
    out["kind"] = kind
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for tag, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(warmup):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[tag] = n_rays / (ms * 1e-3)
            out[tag + "_ms_per_step"] = ms
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out["note"] = "same config, same step definition, eager PyTorch on the same B200, %d steps after %d warm-up" % (steps, warmup)
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    n_rays = cfg["B"] * (cfg["rand_rays"] // cfg["B"])
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.device == "cuda":
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
        tgb = torch_gpu_baseline(args.config, dev, steps=args.steps, warmup=max(args.warmup, 1))
        v, kind, cores, dt = tgb["fp32"], tgb["kind"], 0, tgb["fp32_ms_per_step"] * 1e-3
        sample = "each step = the full batch on the GPU (eager PyTorch fp32, TF32 off); tf32: %.0f rays/s" % tgb["tf32"]
    else:
        step, kind = reference_step_fn(args.config, torch.device("cpu"))
        cores, tried = pick_cpu_threads(step)
        for _ in range(max(0, min(args.warmup, 1))):
            step()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
        dt = (time.perf_counter() - t0) / args.steps
        v = n_rays / dt
        sample = "each step = the full batch of config %s (%d rays), fwd + loss + bwd; thread counts tried (s/step): %s" % (args.config, n_rays, tried)
    line = dict(impl="reference", metric=METRIC, value=v, unit="rays/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling=cfg["scaling"], vs_baseline=None,
                dtype="fp32 (torch CPU)" if args.device != "cuda" else "fp32 (torch CUDA, TF32 off)", data="synthetic",
                config=dict(workload=cfg["desc"], name=args.config, rays_per_gpu=n_rays, global_rays=n_rays,
                            samples_per_ray=cfg["S"], fine_samples_per_ray=(cfg["S"] + cfg["S_fine"]) if cfg["fine"] else 0,
                            note="timed on the torch restatement oracle/sparf_oracle.py, pinned to the reference by tests/golden"),
                cpu_baseline=dict(value=v, unit="rays/s", cores=cores, kind=kind, sample=sample),
                e2e=dict(value=v, unit="rays/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=list(CONFIGS))
    ap.add_argument("--engine", default="auto")
    ap.add_argument("--sync-each-step", type=int, default=1,
                    help="1 (default): synchronise after every timed step, each step starts on an idle device; 0: the K "
                         "steps are enqueued back to back (measured ~1 %% slower on a power-capped B200: lower clocks)")
    ap.add_argument("--device", default="cpu", choices=["cpu", "cuda"], help="reference arm only")
    ap.add_argument("--graph", type=int, default=1, help="1: replay the step as one CUDA graph (default), 0: eager")
    ap.add_argument("--allreduce-in-graph", type=int, default=1)
    ap.add_argument("--no-baselines", action="store_true", help="skip the cpu_baseline / torch_gpu_baseline legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, gradients and render outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to --impl ours")
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
