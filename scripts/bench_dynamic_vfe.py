"""DynamicMeanVFE timing (ops.voxelize_dynamic) on the bench batch (four nus_0075 frames, collated) and on four waymo_010
frames, next to the hard voxelizer + MeanVFE (ops.voxelize + ops.mean_vfe, the bench's caps) on the same batch.  Kernel
times from torch.profiler (CUDA activity, a run of its own), whole calls from a host clock around a call that ends in a
synchronise with the L2 flushed before each, the two paths alternated in one process; the points-per-voxel distribution
that sizes the short (thread) and long (CTA) paths; prints the card's name and power limit and writes a markdown table
(committed as profiles/r07_dynamic_vfe.md).

    python scripts/bench_dynamic_vfe.py [--out PATH]
"""
import argparse, json, os, re, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile
from toda_b200 import ops, synth

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="profiles/r07_dynamic_vfe.md")
args = ap.parse_args()

dev = torch.device("cuda", 0)
peak = 7700.0
if os.path.exists("MEASURED_PEAKS.json"):
    peak = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"]
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
ITERS = 20


def segment_stats(collated, cfg):
    lo, vs = np.float32(cfg["pc_range"][:3]), np.float32(cfg["voxel_size"])
    grid = ops.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    with np.errstate(invalid="ignore"):
        q = np.floor((collated[:, 1:4] - lo) / vs)
    keep = np.all((q >= 0) & (q < grid), axis=1)
    c = np.concatenate([collated[keep, :1], q[keep]], 1).astype(np.int64)
    key = ((c[:, 0] * grid[0] + c[:, 1]) * grid[1] + c[:, 2]) * grid[2] + c[:, 3]
    cnt = np.unique(key, return_counts=True)[1]
    edges = [(1, 1), (2, 3), (4, 8), (9, 32), (33, 1 << 30)]
    hist = {f"{a}" if a == b else (f"{a}-{b}" if b < 1 << 30 else f">{a - 1}"): int(((cnt >= a) & (cnt <= b)).sum())
            for a, b in edges}
    return dict(V=int(cnt.size), max=int(cnt.max()), p99=float(np.percentile(cnt, 99)), mean=float(cnt.mean()), hist=hist)


def kernel_table(fn):
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(ITERS):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
    rows = {}
    for ev in prof.key_averages():
        if ev.self_device_time_total > 0 and "fill" not in ev.key and "elementwise" not in ev.key:
            name = re.sub(r"\(.*$", "", ev.key.replace("(anonymous namespace)::", ""))
            t, c = rows.get(name, (0.0, 0.0))
            rows[name] = (t + ev.self_device_time_total / ITERS, c + ev.count / ITERS)
    return rows


def run(config, batch=4):
    cfg = synth.CONFIGS[config]
    frames, collated = synth.make_batch(config, batch)
    pts = torch.from_numpy(collated).to(dev)
    offs = torch.tensor(np.cumsum([0] + [f.shape[0] for f in frames]), dtype=torch.int32, device=dev)
    pcr, vs = cfg["pc_range"], cfg["voxel_size"]
    k, mv = cfg["max_points"], cfg["max_voxels"]["train"]

    def dynamic():
        return ops.voxelize_dynamic(pts, offs, pcr, vs)

    def hard():
        v, c, num, _ = ops.voxelize(pts, offs, pcr, vs, k, mv, xyz_col=1, feat_col=1, order=ops.ORDER_CANONICAL)
        return ops.mean_vfe(v, num), c

    f, c, counts = dynamic()
    hard()
    ops.reset_launches()
    dynamic()
    launches = ops.launches()
    ts = {"dynamic": [], "hard": []}
    for it in range(2 * ITERS + 6):
        name, fn = ("dynamic", dynamic) if it % 2 == 0 else ("hard", hard)
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        if it >= 6:
            ts[name].append((time.perf_counter() - t0) * 1e6)
    n, stride = pts.shape
    v, nf = f.shape
    seg = segment_stats(collated, cfg)
    assert seg["V"] == v
    return dict(config=config, n=n, stride=stride, V=v, F=nf, launches=launches, seg=seg,
                call_us={k2: float(np.median(x)) for k2, x in ts.items()},
                kernels_dynamic=kernel_table(dynamic), kernels_hard=kernel_table(hard),
                bytes=4.0 * stride * n + 4.0 * nf * v + 16.0 * v, k=k, mv=mv)


card = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                       "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
results = [run("nus_0075"), run("waymo_010")]

lines = ["# DynamicMeanVFE on the device (ops.voxelize_dynamic)", "",
         f"Card: {card} (name, power limit), read in the same run.  `scripts/bench_dynamic_vfe.py`.  Kernel times: "
         f"torch.profiler, mean of {ITERS} calls, L2 flushed before each call.  Whole calls: host clock around a call that "
         f"ends in a synchronise, L2 flushed before each, median of {ITERS}, the dynamic path and hard voxelization + "
         "MeanVFE (`ops.voxelize` with the workload's caps, canonical order, then `ops.mean_vfe`) alternated.", ""]
for r in results:
    s = r["seg"]
    dyn_us = sum(t for t, _ in r["kernels_dynamic"].values())
    hard_us = sum(t for t, _ in r["kernels_hard"].values())
    gbs = r["bytes"] / dyn_us / 1e3 if dyn_us else 0.0
    lines += [f"## {r['config']}: four frames, {r['n']} points, stride {r['stride']}", "",
              f"V = {r['V']} voxels, F = {r['F']}.  Points per voxel: max {s['max']}, p99 {s['p99']:.0f}, mean {s['mean']:.2f}; "
              "voxels by points: " + ", ".join(f"{k}: {v}" for k, v in s["hist"].items()) + ".  "
              f"Launches of one dynamic call (toda_launch_count): {r['launches']}.", "",
              "| path | whole call, us (host clock) | kernel sum, us (profiler) |", "|---|---|---|",
              f"| voxelize_dynamic | {r['call_us']['dynamic']:.1f} | {dyn_us:.1f} |",
              f"| voxelize (K={r['k']}, max_voxels={r['mv']}) + mean_vfe | {r['call_us']['hard']:.1f} | {hard_us:.1f} |", "",
              f"Dynamic path algorithmic bytes (4*stride*N read + 4*F*V + 16*V written) = {r['bytes'] / 1e6:.1f} MB over "
              f"{dyn_us:.1f} us of kernel time = {gbs:.0f} GB/s, {100 * gbs / peak:.1f}% of {peak:.0f} GB/s HBM.", "",
              "| voxelize_dynamic launch | us per call | launches per call |", "|---|---|---|"]
    lines += [f"| {k} | {t:.1f} | {c:g} |" for k, (t, c) in sorted(r["kernels_dynamic"].items(), key=lambda kv: -kv[1][0])]
    lines += ["", "| voxelize + mean_vfe launch | us per call | launches per call |", "|---|---|---|"]
    lines += [f"| {k} | {t:.1f} | {c:g} |" for k, (t, c) in sorted(r["kernels_hard"].items(), key=lambda kv: -kv[1][0])]
    lines.append("")
text = "\n".join(lines)
print(text)
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
open(args.out, "w").write(text)
