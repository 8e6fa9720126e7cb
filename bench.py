#!/usr/bin/env python
"""bench.py -- frames/s of the hot path on B200 (BASELINE.json metric), one JSON line on stdout.

Workload (config.workload): BASELINE.json configs[2] -- "CenterPoint VoxelResBackBone8x fwd+bwd, nuScenes
0.075 m grid 1440x1440x41, batch 4/GPU": one step = hard-voxelize 4 synthetic nuScenes-shaped 10-sweep frames
(K1) -> MeanVFE (K2) -> rulebooks (K3/K4) -> VoxelResBackBone8x forward, train-mode BatchNorm (K5/K8) ->
HeightCompression (K9) -> backward to voxel_features and every parameter (K6/K7/K8) -> gradient all-reduce
(N>1 only).  `value` = frames/s with the points resident in HBM; `e2e` = the same step fed from pinned HOST
memory through the plugin modules, H2D copy and a D2H read of the loss inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision fp32|bf16] [--dump-outputs DIR]
Under torchrun every rank runs its own 4 frames (weak scaling); rank 0 prints the line.
--dump-outputs DIR writes what the last timed step of the device-resident arm computed (rank 0) as DIR/<name>.npy, so that
two builds can be compared output for output on identical seeded inputs (see dump_outputs()).
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

# stdout must carry exactly ONE JSON line, but libraries (NCCL's version banner, ...) print there too: keep a private
# handle on the real stdout for the result and point fd 1 at stderr for everything else
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


# Row counts differ from batch to batch, so every step asks the caching allocator for slightly different sizes; with exact
# sizes the freed blocks of one batch rarely fit the next, the pools fragment and torch falls back to cudaMalloc inside a
# timed step (which stalls for as long as the GPU's queue: seen as single 40-70 ms steps).  Rounding request sizes to 1/8
# power-of-two steps maps successive batches onto the same size classes.  (Standard PyTorch allocator option; must be
# set before the first CUDA allocation.  INTEGRATION.md recommends the same for training runs.)
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "roundup_power2_divisions:8")

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from toda_b200 import synth  # noqa: E402

FRAMES_PER_GPU = 4
POOL = 3                     # distinct pre-staged batches rotated through, so no step re-reads a warm input
# The default line is BASELINE.json configs[2]; the other configs are measured with --workload and never replace it.
WORKLOADS = {
    "nus_0075": dict(cfg="nus_0075", net="VoxelResBackBone8x", train=True, metric="frames/s voxelize+VoxelResBackBone8x fwd+bwd",
                     desc="BASELINE.json configs[2]: CenterPoint VoxelResBackBone8x fwd+bwd, nuScenes-shaped 10-sweep frames, 0.075 m "
                          "voxels, grid 1440x1440x41, batch 4/GPU, train-mode BN, K=10, max_voxels 120000"),
    "waymo_second": dict(cfg="waymo_010", net="VoxelBackBone8x", train=False, metric="frames/s voxelize+VoxelBackBone8x fwd",
                         desc="BASELINE.json configs[1]: SECOND VoxelBackBone8x forward (eval-mode BN), Waymo-shaped frames, 0.1 m "
                              "voxels, grid 1504x1504x41, batch 4/GPU, K=5, max_voxels 150000"),
    "toda_stage2": dict(cfg="toda_stage2", net="VoxelResBackBone8x", train=True, mixed=True,
                        metric="frames/s voxelize+VoxelResBackBone8x fwd+bwd (TODA stage-2 batch)",
                        desc="BASELINE.json configs[3]: TODA stage-2 step, batch of 4 = 2 intra-domain mixups + 2 Waymo/nuScenes polar "
                             "sector swaps (mixed on the host side of the timer), CenterPoint VoxelResBackBone8x fwd+bwd, grid "
                             "1440x1440x50 (z -5..4.8), F=4, 1 sweep, K=10, max_voxels 120000"),
}
WORKLOAD = "nus_0075"
METRIC = WORKLOADS[WORKLOAD]["metric"]


class Cfg(dict):
    __getattr__ = dict.get


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region through NVML (a polling thread; a concurrent
    `nvidia-smi -lms` process was seen to stall the driver for tens of ms inside single steps).  Falls back to one
    nvidia-smi query if NVML cannot be loaded."""

    def __init__(self, index, period_s=0.02):
        self.sm, self.max_sm, self.reasons, self.nv = [], None, set(), None
        self._stop = threading.Event()
        self.recording = False        # the thread polls from start-up (NVML's first calls are slow); samples count only
                                      # between begin() and stop(), i.e. inside the timed region
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            phys, vis = index, os.environ.get("CUDA_VISIBLE_DEVICES", "")
            parts = [x.strip() for x in vis.split(",")] if vis else []
            if parts and all(x.isdigit() for x in parts) and index < len(parts):
                phys = int(parts[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.period = period_s
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        names = {getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                 getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                 getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap"}
        while not self._stop.is_set():
            try:
                clk = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.recording:
                    self.sm.append(clk)
                    for bit, nm in names.items():
                        if mask & bit:
                            self.reasons.add(nm)
            except Exception:
                pass
            self._stop.wait(self.period)

    def begin(self):
        self.recording = True

    def stop(self):
        self.recording = False
        if self.nv is not None:
            self._stop.set()
            self.t.join(timeout=1.0)
            if self.sm:
                return dict(sm_mhz=float(np.median(self.sm)), sm_max_mhz=self.max_sm, reasons=sorted(self.reasons),
                            samples=len(self.sm), source="nvml")
        try:
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            out = subprocess.check_output(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits"], text=True,
                                          timeout=10).strip().splitlines()[0]
            f = [x.strip() for x in out.split(",")]
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            return dict(sm_mhz=float(f[0]), sm_max_mhz=float(f[1]), samples=1, source="nvidia-smi (after the timed region)",
                        reasons=[n for n, v in zip(names, f[2:6]) if v.lower().startswith("active")])
        except Exception:
            return None


# ---------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------
def build_hot_path(device, precision):
    import toda_b200.pcdet_plugin as P
    from toda_b200.spconv_compat import pytorch as sp
    sp.set_conv_precision(precision)
    wl = WORKLOADS[WORKLOAD]
    cfg = synth.CONFIGS[wl["cfg"]]
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    torch.manual_seed(666)   # the reference's --fix_random_seed value
    vfe = P.MeanVFE(Cfg(MAX_POINTS_PER_VOXEL=cfg["max_points"], MAX_NUMBER_OF_VOXELS=cfg["max_voxels"]), cfg["num_features"],
                    voxel_size=cfg["voxel_size"], point_cloud_range=cfg["pc_range"], grid_size=grid)
    net = getattr(P, wl["net"])(Cfg(), cfg["num_features"], grid)
    hc = P.HeightCompression(Cfg(NUM_BEV_FEATURES=256))
    for m in (vfe, net, hc):
        m.to(device).train(wl["train"])
    return vfe, net, hc


def _stage2_frames(first, device):
    """Four stage-2 samples (BASELINE configs[3]): two intra-domain mixups (intra_domain_point_mixup.py L15-72, lam ~
    Beta(2,2)) and two polar sector swaps of a Waymo-shaped frame into a nuScenes-shaped one (inter_domain_point_polarmix.py
    L72-95, pi/2 sector), built once, outside the timer, with the K0 point kernels; the reference mixes in its dataset
    workers, i.e. also on the input side of the step."""
    from toda_b200.pcdet_plugin import processor as GP
    f = synth.CONFIGS["toda_stage2"]["num_features"]
    rng = np.random.default_rng(40000 + first)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a[:, :f])).to(device)    # noqa: E731
    out = []
    for i in range(FRAMES_PER_GPU):
        a = synth.make_frame("toda_stage2", first * 3 + 3 * i)
        if i % 2 == 0:
            b = synth.make_frame("toda_stage2", first * 3 + 3 * i + 1)
            lam = float(rng.beta(2.0, 2.0))
            m = GP.mixup_points(t(a), t(b), lam, rng.permutation(a.shape[0]), rng.permutation(b.shape[0]))
        else:
            w = synth.make_frame("waymo_010", first + i)
            s0 = float(rng.random() * np.pi * 2 - np.pi)
            m = GP.polar_swap_points(t(a), t(w), s0, s0 + np.pi / 2)
        out.append(m.cpu().numpy())
    return out


def host_batches(rank, n_batches, device=None):
    """Pinned host copies of collated `points` [b,x,y,z,...] (dataset.py L173-178) + frame offsets."""
    wl = WORKLOADS[WORKLOAD]
    out = []
    for j in range(n_batches):
        first = (rank * POOL + j) * FRAMES_PER_GPU
        if wl.get("mixed"):
            frames = _stage2_frames(first, device)
            collated = np.concatenate([np.pad(f, ((0, 0), (1, 0)), mode="constant", constant_values=i) for i, f in enumerate(frames)])
        else:
            frames, collated = synth.make_batch(wl["cfg"], FRAMES_PER_GPU, first_frame=first)
        offs = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)
        out.append((torch.from_numpy(np.ascontiguousarray(collated, dtype=np.float32)).pin_memory(), torch.from_numpy(offs).pin_memory()))
    return out


def run_ours(args, rank, world, local_rank):
    from toda_b200 import ops
    from toda_b200.dist import FlatGradBucket
    from toda_b200.pipeline import InputPipeline
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    vfe, net, hc = build_hot_path(device, args.precision)
    bucket = FlatGradBucket(net.parameters())
    train = WORKLOADS[WORKLOAD]["train"]
    hosts = host_batches(rank if args.data_rank is None else args.data_rank, POOL, device)
    devs = [(p.to(device), o.to(device)) for p, o in hosts]
    cot = None

    trace = [] if os.environ.get("TODA_BENCH_TRACE") else None

    def step(points, offsets, reduce=True):
        nonlocal cot
        t0 = time.perf_counter()
        bucket.zero()
        bd = {"points": points, "point_frame_offsets": offsets, "batch_size": FRAMES_PER_GPU}
        with torch.set_grad_enabled(train):
            bd = vfe(bd)
            t1 = time.perf_counter()
            bd = hc(net(bd))
        t2 = time.perf_counter()
        sf = bd["spatial_features"]
        if cot is None:
            cot = torch.randn(sf.shape, device=device, generator=torch.Generator(device=device).manual_seed(1)) / sf.numel()
        loss = (sf * cot).sum()
        if train:
            loss.backward()
            if reduce:
                bucket.all_reduce_mean()
        if trace is not None:
            t3 = time.perf_counter()
            trace.append((round((t1 - t0) * 1e3, 2), round((t2 - t1) * 1e3, 2), round((t3 - t2) * 1e3, 2)))
        return loss, bd

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm -----------------------------------------------------------------------------
    # priming (untimed, before the W warm-up steps): reserve a large cached block once (row counts differ from batch to
    # batch, and the caching allocator must never fall back to a device-synchronising cudaMalloc / cudaFree in a timed
    # step), then every pooled batch twice so that workspace growth and cudaFuncSetAttribute are behind us
    sampler = ClockSampler(local_rank) if rank == 0 else None
    reserve = torch.empty(24 << 30, dtype=torch.uint8, device=device)
    del reserve
    for i in range(2 * POOL):
        step(*devs[i % POOL])
    barrier()
    # The cyclic GC stays enabled (with it disabled, step garbage pins ~5 GB of activations per step and the allocator
    # falls back to cudaMalloc).  gc.freeze() moves the long-lived heap (torch, numpy, modules: ~1 M objects) to the
    # permanent generation so that the full collections that fall inside the timed region only walk the young objects
    # of the steps -- without it a gen-2 pass over the whole heap shows up as one 20-90 ms step.
    gc.collect()
    gc.freeze()
    # ---- pipelined steps (what is timed) -------------------------------------------------------------------
    # One step = the backbone fwd+bwd (+ gradient all-reduce) of batch i on the main stream, then the front of batch i+1
    # (voxelize, MeanVFE, index + rulebooks of every level; in the e2e arm also its H2D copy) submitted to the input
    # pipeline's side stream, where it overlaps with the kernels just queued.  Every timed step therefore contains
    # exactly one front and one fwd+bwd; only the pipeline fill (the front of the first batch) precedes the timer, as
    # a DataLoader's prefetch would.
    pipe = InputPipeline(vfe, net, device)

    host = dict(front=0.0, back=0.0)     # host wall time inside the two halves of a step (front includes its small device waits)

    def front(points, offsets, pending):
        t0 = time.perf_counter()
        if trace is not None:
            import faulthandler
            faulthandler.dump_traceback_later(0.012, file=sys.stderr)     # where is the host if a front stalls?
        h = pipe.submit({"points": points, "point_frame_offsets": offsets, "batch_size": FRAMES_PER_GPU},
                        inputs_pending=pending)
        host["front"] += time.perf_counter() - t0
        if trace is not None:
            faulthandler.cancel_dump_traceback_later()
            trace.append(("front", round((time.perf_counter() - t0) * 1e3, 2)))
        return h

    def back(handle, reduce=True):
        t0 = time.perf_counter()
        bucket.zero()
        with torch.set_grad_enabled(train):
            bd = hc(net(pipe.consume(handle)))
        t1 = time.perf_counter()
        loss = (bd["spatial_features"] * cot).sum()
        if train:
            loss.backward()
            if reduce:
                bucket.all_reduce_mean()
        host["back"] += time.perf_counter() - t0
        if trace is not None:
            trace.append(("back", round((t1 - t0) * 1e3, 2), round((time.perf_counter() - t1) * 1e3, 2)))
        return loss, bd

    if trace is not None:
        gc_t = {}

        def gc_cb(phase, info):
            if phase == "start":
                gc_t["t"] = time.perf_counter()
            else:
                trace.append(("gc", info["generation"], info["collected"], round((time.perf_counter() - gc_t["t"]) * 1e3, 2)))
        gc.callbacks.append(gc_cb)

    h = front(*devs[0], False)
    for i in range(2 * POOL + args.warmup):   # every pooled batch twice through the pipeline (side-stream pool), then W warm-up steps
        loss, bd = back(h)
        h = front(*devs[(i + 1) % POOL], False)
    barrier()
    if sampler:
        sampler.begin()
    ops.reset_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    mark0 = len(trace) if trace is not None else 0
    host["front"] = host["back"] = 0.0
    e0.record()
    marks[0].record()
    for i in range(args.steps):
        loss, bd = back(h)
        h = front(*devs[(2 * POOL + args.warmup + i + 1) % POOL], False)   # pre-staged, complete device tensors
        marks[i + 1].record()
    torch.cuda.current_stream().wait_stream(pipe.stream)        # the last front belongs to the timed region too
    e1.record()
    barrier()                       # (also drains the side stream: torch.cuda.synchronize)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, bd, net)
    per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(args.steps)]
    if rank == 0:
        print("per-step ms (device arm, main stream): " + " ".join("%.2f" % t for t in per_step), file=sys.stderr)
        if trace is not None:
            print("host trace (ms) of the timed steps: " + " ".join(str(t) for t in trace[mark0:]), file=sys.stderr)
    ms = e0.elapsed_time(e1)
    launches = ops.launches()
    host_ms = dict(fwd_bwd=host["back"] * 1e3 / args.steps, front=host["front"] * 1e3 / args.steps)
    t = torch.tensor([ms], device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * FRAMES_PER_GPU * args.steps / (ms / 1e3)

    # ---- end-to-end arm: pinned host points -> H2D -> front -> fwd+bwd -> D2H loss, same pipeline ------------
    def e2e_step(h, i):
        loss, _ = back(h)
        hp, ho = hosts[(i + 1) % POOL]
        nxt = front(hp, ho, False)                   # H2D of the next batch from pinned memory, on the side stream
        return float(loss.item()), nxt               # D2H read of this step's result
    h = front(*hosts[0], False)
    # (the H2D path and its side-pool size classes warm up too: every pre-staged batch is copied at least once more than
    # the pool holds, so that no first-time allocation of a staging tensor -- a cudaMalloc, i.e. a device-wide sync of
    # ~50 ms, seen as one outlier step in 2 of ~40 runs -- can land in the timed region)
    for i in range(max(POOL + 2, args.warmup)):
        _, h = e2e_step(h, i)
    barrier()
    e0.record()
    wall = [time.perf_counter()]
    mark1 = len(trace) if trace is not None else 0
    for i in range(args.steps):
        _, h = e2e_step(h, i)
        wall.append(time.perf_counter())
    torch.cuda.current_stream().wait_stream(pipe.stream)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    if rank == 0:
        print("per-step ms (e2e arm, host wall clock): " + " ".join("%.2f" % ((b - a) * 1e3) for a, b in zip(wall, wall[1:])),
              file=sys.stderr)
        if trace is not None:
            print("host trace (ms) of the e2e steps: " + " ".join(str(t) for t in trace[mark1:]), file=sys.stderr)
    h2d = int(np.mean([p.numel() * 4 + o.numel() * 4 for p, o in hosts]))
    e2e = dict(value=world * FRAMES_PER_GPU * args.steps / (e2e_ms / 1e3), unit="frames/s", h2d_bytes_per_step=h2d,
               d2h_bytes_per_step=4 * 6, ms_per_step=e2e_ms / args.steps)
    del h

    if rank != 0:
        return None
    # ---- roofline pass (rank 0): per-call device times of one more step, not part of `value` ----------------
    peaks = load_peaks()
    with bucket.no_sync():                      # rank 0 only: the gradient hooks must not launch a collective here
        step(*devs[0], reduce=False)            # (re-warms the allocator for the in-line call sequence)
        torch.cuda.synchronize()
        ops.profile_begin()
        loss, bd = step(*devs[0], reduce=False)
        prof = ops.profile_end()
    roof, layers = roofline_from_profile(prof, bd, peaks, ms / args.steps)
    line = dict(metric=WORKLOADS[WORKLOAD]["metric"], value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype={"fp32": "f32", "bf16": "bf16", "bf16x3": "bf16x3 (split bf16, fp32-class)"}[args.precision], data="synthetic",
                config=dict(conv_kernel="row-cache / TMEM-operand (conv_ts.cu, opt-in)" if ops.tile_plans_enabled() else "round-1 tcgen05 kernels (conv_tc.cu / conv_tma.cu)",
                            workload=WORKLOADS[WORKLOAD]["desc"], workload_key=WORKLOAD,
                            frames_per_gpu=FRAMES_PER_GPU, points_per_frame=int(hosts[0][0].shape[0] / FRAMES_PER_GPU),
                            voxels_per_frame=int(bd["voxel_coords"].shape[0] / FRAMES_PER_GPU), conv_precision=args.precision,
                            l2="inputs rotate over %d pre-staged batches and each step streams >1 GB of activations (>> 126 MB L2)" % POOL,
                            parallelism=f"dp{world} (frame-sharded" + (", bucketed grad all-reduce overlapped with backward)" if train else ", no collective: forward only)")),
                clocks=clocks, e2e=e2e, gpu_launches=int(launches), launches_per_step=launches / args.steps,
                host_ms_per_step=round(host_ms["fwd_bwd"] + host_ms["front"], 3),
                host_ms_detail=dict(fwd_bwd=round(host_ms["fwd_bwd"], 3), front_incl_device_waits=round(host_ms["front"], 3)),
                roofline=roof, roofline_layers=layers)
    return line


DUMP_BYTES = 64 << 20       # cap on everything dump_outputs() writes


def dump_outputs(out_dir, loss, bd, net):
    """What a caller of the timed step receives, as float32 / float64 .npy files in `out_dir`:
      loss.npy                          the step's scalar loss (float64)
      grad.<parameter name>.npy         every parameter gradient of the backbone (train workloads), full
      spatial_features_channel_sum.npy  the dense BEV map summed over H x W per (frame, channel), float64, full coverage
      spatial_features_sample.npy       the dense BEV map [B, C, H, W] at a fixed sample of flat positions (drawn with
                                        numpy.random.default_rng(0), sorted), as many as fit in what is left of DUMP_BYTES
    The sparse tensors are left out: their row order is an implementation detail, the dense BEV map is not."""
    os.makedirs(out_dir, exist_ok=True)
    sf = bd["spatial_features"].detach()
    arrays = {"loss": np.asarray(float(loss.item()), dtype=np.float64),
              "spatial_features_channel_sum": sf.double().sum(dim=(2, 3)).cpu().numpy()}
    for name, p in net.named_parameters():
        if p.grad is not None:
            arrays["grad." + name] = p.grad.detach().float().cpu().numpy()
    left = (DUMP_BYTES - (1 << 20) - sum(a.nbytes for a in arrays.values())) // 4     # 1 MB kept for the .npy headers
    if left <= 0:
        raise RuntimeError("dump_outputs: gradients alone exceed %d bytes" % DUMP_BYTES)
    n = sf.numel()
    if n <= left:
        arrays["spatial_features_sample"] = sf.float().reshape(-1).cpu().numpy()
    else:
        idx = np.sort(np.random.default_rng(0).choice(n, size=left, replace=False))
        arrays["spatial_features_sample"] = sf.float().reshape(-1)[torch.from_numpy(idx).to(sf.device)].cpu().numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    print("dumped %d arrays (%.1f MB) to %s" % (len(arrays), sum(a.nbytes for a in arrays.values()) / 2**20, out_dir), file=sys.stderr)


def roofline_from_profile(prof, bd, peaks, step_ms):
    """Algorithmic flops / bytes per call (SURVEY.md section 8d formulas) over the measured call durations."""
    from collections import defaultdict
    pairs_cache = {}

    def pairs_of(rb_id):
        return pairs_cache.get(rb_id)
    # pair counts per rulebook (computed outside any timed region)
    for key, (rb, _) in bd["encoded_spconv_tensor"].indice_dict.items():
        pairs_cache[id(rb)] = int((rb.nbr_fwd >= 0).sum().item())
    groups = defaultdict(lambda: dict(ms=0.0, calls=0, flops=0.0, bytes=0.0))
    for r in prof:
        name = r["name"]
        g = None
        if name in ("conv_fwd", "conv_dgrad", "conv_wgrad"):
            P = pairs_of(r["rb"]) or 0
            e = 4 if r["precision"] == 0 else 2
            flops = 2.0 * P * r["cin"] * r["cout"]
            byts = e * (r["n_in"] * r["cin"] + r["n_out"] * r["cout"]) + 8.0 * P + e * r["kvol"] * r["cin"] * r["cout"]
            key = f"{name} {r['cin']}->{r['cout']} k{r['kvol']}"
            g = groups[key]
            g["flops"] += flops
            g["bytes"] += byts
            g["kind"] = "conv"
        elif name == "voxelize":
            v = bd["voxel_coords"].shape[0]
            byts = 4.0 * r["n_points"] * r["F"] + 4.0 * v * r["K"] * r["F"] + 16.0 * v + 4.0 * v
            g = groups[name]
            g["bytes"] += byts
            g["kind"] = "hbm"
        elif name in ("bn_apply", "bn_stats", "bn_bwd", "mean_vfe_fwd", "bev_scatter_fwd", "bev_scatter_bwd", "rulebook_subm",
                      "rulebook_sparse", "index_build"):
            g = groups[name]
            g["kind"] = "hbm"
            if name == "bn_apply":
                g["bytes"] += 4.0 * r["n"] * r["c"] * (3 if r["residual"] else 2)
            elif name == "bn_stats":
                g["bytes"] += 4.0 * r["n"] * r["c"]
            elif name == "bn_bwd":
                g["bytes"] += 4.0 * r["n"] * r["c"] * (8 if r["residual"] else 7)
            elif name == "mean_vfe_fwd":
                g["bytes"] += 4.0 * r["V"] * r["K"] * r["F"] + 4.0 * r["V"] + 4.0 * r["V"] * r["F"]
            elif name == "bev_scatter_fwd":
                g["bytes"] += 4.0 * r["n"] * r["c"] + 16.0 * r["n"] + 4.0 * r["out_elems"]
            elif name == "bev_scatter_bwd":
                g["bytes"] += 8.0 * r["n"] * r["c"] + 16.0 * r["n"]
            elif name == "rulebook_subm":
                g["bytes"] += 16.0 * r["n"] + 4.0 * r["kvol"] * r["n"]
            elif name == "rulebook_sparse":
                g["bytes"] += 16.0 * (r["n_in"] + r["n_out"]) + 4.0 * r["kvol"] * (r["n_in"] + r["n_out"])
        if g is not None:
            g["ms"] += r["ms"]
            g["calls"] += 1
    total_ms = sum(g["ms"] for g in groups.values())
    layers = []
    for key, g in sorted(groups.items(), key=lambda kv: -kv[1]["ms"]):
        row = dict(kernel=key, calls=g["calls"], ms=round(g["ms"], 4), share_of_profiled=round(g["ms"] / max(total_ms, 1e-9), 4))
        if g["ms"] > 0:
            if g.get("kind") == "conv":
                row["tflops"] = round(g["flops"] / (g["ms"] * 1e-3) / 1e12, 3)
                row["frac_of_bf16_peak"] = round(row["tflops"] / peaks["bf16_tflops_sustained"], 5)
                row["gbs"] = round(g["bytes"] / (g["ms"] * 1e-3) / 1e9, 1)
            elif g["bytes"] > 0:
                row["gbs"] = round(g["bytes"] / (g["ms"] * 1e-3) / 1e9, 1)
                row["frac_of_hbm_peak"] = round(row["gbs"] / peaks["hbm_gbs"], 4)
        layers.append(row)
    # dominant KERNEL (device function): forward and dgrad convolutions are the same tcgen05 kernel
    # (conv_ts_fwd_kernel, csrc/conv_ts.cu), the weight gradient is conv_tc_wgrad_kernel
    from toda_b200 import ops as _ops
    fwd_kernel = "conv_ts_fwd_kernel" if _ops.tile_plans_enabled() else "conv_tc_fwd_kernel"
    fams = defaultdict(lambda: dict(ms=0.0, calls=0, flops=0.0, bytes=0.0, kind="hbm"))
    for key, g in groups.items():
        fam = (fwd_kernel + " (fwd + dgrad, all layers)" if key.startswith(("conv_fwd", "conv_dgrad")) else
               "conv_tc_wgrad_kernel (all layers)" if key.startswith("conv_wgrad") else key)
        f = fams[fam]
        for k in ("ms", "calls", "flops", "bytes"):
            f[k] += g[k]
        f["kind"] = g.get("kind", "hbm")
    top_key, top = max(fams.items(), key=lambda kv: kv[1]["ms"])
    traffic = None
    # dram bytes per launch from the committed ncu --set full captures (r02: conv_ts_fwd_kernel + wgrad; r01: conv_tc_fwd_kernel)
    for tname in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if traffic is None and os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(top_key.split(" ")[0])
    if top.get("kind") == "conv":
        achieved = top["flops"] / (top["ms"] * 1e-3) / 1e12
        roof = dict(bound="tensor", kernel=top_key, achieved=achieved, peak=peaks["bf16_tflops_sustained"], unit="TFLOP/s",
                    frac=achieved / peaks["bf16_tflops_sustained"], traffic=traffic,
                    peak_source=peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    launches=top["calls"], avg_launch_ms=top["ms"] / top["calls"], share_of_step=top["ms"] / step_ms,
                    flops_per_launch=top["flops"] / top["calls"], algorithmic_bytes_per_launch=top["bytes"] / top["calls"])
    else:
        achieved = top["bytes"] / (top["ms"] * 1e-3) / 1e9
        roof = dict(bound="hbm", kernel=top_key, achieved=achieved, peak=peaks["hbm_gbs"], unit="GB/s", frac=achieved / peaks["hbm_gbs"],
                    traffic=traffic, peak_source=peaks["source"], launches=top["calls"], avg_launch_ms=top["ms"] / top["calls"],
                    share_of_step=top["ms"] / step_ms, algorithmic_bytes_per_launch=top["bytes"] / top["calls"])
    return roof, layers


# ---------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's path, on the host cores
# ---------------------------------------------------------------------------------------------------------------
def cpu_step_time(n_frames, steps, warmup):
    """Seconds per step of the CPU path on `n_frames` full-size frames: voxelize (C restatement of the
    Point2VoxelCPU3d loop, one thread per frame as a DataLoader worker would) + MeanVFE + VoxelResBackBone8x
    fwd+bwd + HeightCompression through the oracle's pure-PyTorch sparse conv (all host threads)."""
    from oracle import voxelize as OV
    from tests import parity_utils as PU
    cfg = synth.CONFIGS[WORKLOADS[WORKLOAD]["cfg"]]
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    torch.manual_seed(666)
    net = PU.oracle_backbones()["VoxelResBackBone8x"](Cfg(), cfg["num_features"], grid)
    net.train()
    gens = [OV.Point2VoxelCPU3d(cfg["voxel_size"], cfg["pc_range"], cfg["num_features"], cfg["max_points"], cfg["max_voxels"]["train"])
            for _ in range(n_frames)]
    frames = [synth.make_frame(WORKLOADS[WORKLOAD]["cfg"], i) for i in range(n_frames)]
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        outs = [[t.numpy() for t in g.point_to_voxel(OV.from_numpy(f))] for g, f in zip(gens, frames)]
        voxels = np.concatenate([o[0] for o in outs])
        num = np.concatenate([o[2] for o in outs])
        coords = np.concatenate([np.pad(o[1], ((0, 0), (1, 0)), constant_values=b) for b, o in enumerate(outs)])
        vf = torch.from_numpy(OV.mean_vfe(voxels, num)).requires_grad_(True)
        for p in net.parameters():
            p.grad = None
        bd = PU._oracle_hc(net({"voxel_features": vf, "voxel_coords": torch.from_numpy(coords).float(), "batch_size": n_frames}))
        sf = bd["spatial_features"]
        (sf * (1.0 / sf.numel())).sum().backward()
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return float(np.mean(times)), int(voxels.shape[0])


def run_reference(args, rank, world):
    if rank != 0:
        return None
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sec, nvox = cpu_step_time(1, args.steps, args.warmup)
    value = 1.0 / sec
    cpu = dict(value=value, unit="frames/s", cores=cores, kind="port",
               sample="1 full-size nuScenes-shaped frame per step (of the 4-frame batch): C voxelizer loop + MeanVFE + "
                      "oracle VoxelResBackBone8x fwd+bwd + dense BEV, torch CPU threads=%d; spconv itself is not installable" % cores)
    return dict(metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=sec * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference", config=dict(workload="BASELINE.json configs[2] (same as the GPU arm), one frame per CPU step",
                                              voxels_per_frame=nvox),
                cpu_baseline=cpu, e2e=dict(value=value, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("TODA_CONV_PRECISION", "bf16"), choices=["fp32", "bf16", "bf16x3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--data-rank", type=int, default=None, help="debug: use the synthetic frames rank R of a multi-GPU run would get")
    ap.add_argument("--workload", default="nus_0075", choices=sorted(WORKLOADS),
                    help="default = BASELINE.json configs[2]; waymo_second = configs[1]; toda_stage2 = configs[3]")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (at most 64 MB)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl ours)")
    global WORKLOAD, METRIC
    WORKLOAD = args.workload
    METRIC = WORKLOADS[WORKLOAD]["metric"]
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        line = run_reference(args, rank, world)
        if line is not None:
            emit(line)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: toda_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    line = run_ours(args, rank, world, local_rank)
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and WORKLOAD == "nus_0075":
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            sec, nvox = cpu_step_time(1, 1, 0)
            line["cpu_baseline"] = dict(value=1.0 / sec, unit="frames/s", cores=cores, kind="port",
                                        sample="one full-size frame, one step (%.1f s): C voxelizer loop + MeanVFE + oracle "
                                               "VoxelResBackBone8x fwd+bwd + dense BEV on torch CPU" % sec)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
