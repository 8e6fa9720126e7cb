"""Cost of synchronized BatchNorm (torch.nn.SyncBatchNorm) in the training step of the default workload.

    torchrun --nproc_per_node N scripts/bench_syncbn.py [--steps K] [--warmup W] [--rounds R] [--precision bf16]

Workload: bench.py's default line (BASELINE.json configs[2]: CenterPoint VoxelResBackBone8x fwd+bwd, 4 nuScenes-shaped
frames per GPU, FlatGradBucket gradient average), run with the backbone's BatchNorm1d and with the same backbone after
torch.nn.SyncBatchNorm.convert_sync_batchnorm.  The two variants alternate in blocks of K steps (R rounds), in the same
processes on the same frames, so that other work on the host affects both alike.  Rank 0 prints one JSON line: ms/step of
each variant (median over the rounds and every round's value), the collectives the synchronized BatchNorms issue per step
(counted), and the card's name and power limit.  Needs N >= 2 (with one rank nothing is synchronized).
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import bench  # noqa: E402


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                                       str(torch.cuda.current_device())], text=True, timeout=30).strip()
        name, limit = [s.strip() for s in out.split(",")[:2]]
        return dict(name=name, power_limit=limit)
    except (OSError, subprocess.SubprocessError, ValueError):
        return dict(name=torch.cuda.get_device_name(), power_limit="unknown")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16", "bf16x3"])
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world < 2:
        raise SystemExit("bench_syncbn.py needs torchrun with 2 or more processes: with one rank nothing is synchronized")
    from toda_b200.dist import FlatGradBucket
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    dist.init_process_group("nccl", device_id=device)
    vfe, net, hc = bench.build_hot_path(device, args.precision)
    net_sync = torch.nn.SyncBatchNorm.convert_sync_batchnorm(copy.deepcopy(net)).to(device).train()
    n_bn = sum(isinstance(m, torch.nn.SyncBatchNorm) for m in net_sync.modules())
    variants = {"batchnorm1d": (net, FlatGradBucket(net.parameters())),
                "syncbn": (net_sync, FlatGradBucket(net_sync.parameters()))}
    hosts = bench.host_batches(rank, bench.POOL, device)
    batches = [(p.to(device), o.to(device)) for p, o in hosts]
    cot = {}

    def step(name, i):
        model, bucket = variants[name]
        points, offsets = batches[i % len(batches)]
        bucket.zero()
        bd = hc(model(vfe({"points": points, "point_frame_offsets": offsets, "batch_size": bench.FRAMES_PER_GPU})))
        sf = bd["spatial_features"]
        if sf.shape not in cot:
            cot[sf.shape] = torch.randn(sf.shape, device=device, generator=torch.Generator(device=device).manual_seed(1)) / sf.numel()
        (sf * cot[sf.shape]).sum().backward()
        bucket.all_reduce_mean()

    # collectives per step: the synchronized BatchNorms' all-reduces are the float64 ones (the gradient buckets are fp32)
    counts = {"bn": 0, "other": 0}
    real = dist.all_reduce

    def counting(t, *a, **k):
        counts["bn" if t.dtype == torch.float64 else "other"] += 1
        return real(t, *a, **k)
    dist.all_reduce = counting
    step("syncbn", 0)
    dist.all_reduce = real
    per_step = dict(counts)

    for name in variants:
        for i in range(args.warmup + bench.POOL):
            step(name, i)
    torch.cuda.synchronize()
    dist.barrier()
    times = {name: [] for name in variants}
    for r in range(args.rounds):
        for name in (variants if r % 2 == 0 else list(reversed(list(variants)))):
            torch.cuda.synchronize()
            dist.barrier()
            t0 = time.perf_counter()
            for i in range(args.steps):
                step(name, i)
            torch.cuda.synchronize()
            dist.barrier()
            times[name].append((time.perf_counter() - t0) * 1e3 / args.steps)
    if rank == 0:
        med = {k: float(np.median(v)) for k, v in times.items()}
        line = dict(metric="syncbn_step_ms", workload="BASELINE.json configs[2], 4 frames per GPU, train step incl. gradient average",
                    gpus=world, precision=args.precision, steps=args.steps, warmup=args.warmup, rounds=args.rounds,
                    ms_per_step=med, ms_per_step_rounds={k: [round(x, 3) for x in v] for k, v in times.items()},
                    syncbn_overhead_ms=round(med["syncbn"] - med["batchnorm1d"], 3),
                    syncbn_overhead_pct=round(100 * (med["syncbn"] / med["batchnorm1d"] - 1), 2),
                    sync_batchnorms=n_bn, collectives_per_step=dict(syncbn=per_step["bn"], gradient_buckets=per_step["other"]),
                    card=card())
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
