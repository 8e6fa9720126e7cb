"""Rotate-paste timing on the bench batch (four nus_0075 frames, collated; 40 destination boxes per frame, 40 instance
boxes per frame centred on points of the frame, PolarMix angles [0, U*2pi/3, (U+1)*2pi/3]; the frames are their own
source, as PolarMix runs on one scan).  Kernel times from torch.profiler (CUDA activity), the whole call from a host clock
around a call that ends in a synchronise, the L2 flushed between iterations; prints the card's name and power limit and
writes a markdown table (committed as profiles/r06_rotate_paste.md).

    python scripts/bench_rotate_paste.py [--out PATH]
"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from tests import rotate_paste_oracle as RP
from toda_b200 import synth
from toda_b200.pcdet_plugin.processor import rotate_paste_points

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="profiles/r06_rotate_paste.md")
args = ap.parse_args()

KERNELS = ("rp_member_kernel", "rp_box_rows_kernel", "gts_accept_kernel", "rp_copy_dst_kernel", "rp_paste_kernel")
CLASSES = np.array(["car", "truck", "bus", "pedestrian", "bicycle"])
dev = torch.device("cuda", 0)
peak = 7700.0
if os.path.exists("MEASURED_PEAKS.json"):
    peak = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"]
frames, collated = synth.make_batch("nus_0075", 4)
offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(dev)
pts = torch.from_numpy(collated).to(dev)
rng = np.random.default_rng(3)


def boxes(centres):
    m = centres.shape[0]
    return np.concatenate([centres, np.array([4.5, 1.9, 1.6]) * rng.uniform(0.7, 1.3, (m, 3)), rng.uniform(-np.pi, np.pi, (m, 1)),
                           rng.normal(0, 2, (m, 2))], 1).astype(np.float32)


gt = [boxes(np.c_[rng.uniform(-50, 50, (40, 2)), rng.uniform(-2, 0, (40, 1))]) for _ in frames]
inst = [boxes(f[rng.integers(0, f.shape[0], 40), :3].astype(np.float64)) for f in frames]
gt_names = [CLASSES[rng.integers(0, 5, 40)] for _ in frames]
inst_names = [CLASSES[rng.integers(0, 5, 40)] for _ in frames]
angles = []
for _ in frames:
    u = rng.random()
    angles.append([0.0, u * 2 * np.pi / 3, (u + 1) * 2 * np.pi / 3])


def step():
    return rotate_paste_points(pts, offs, pts, offs, gt, gt_names, inst, inst_names, angles, x_col=1)


flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
out = step()
n_in, n_out, stride = pts.shape[0], out[0].shape[0], pts.shape[1]
acc = sum(b.shape[0] - g.shape[0] for b, g in zip(out[2], gt))
ts = []
for it in range(23):
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step()                                  # synchronises once inside, on the accepted flags and per-frame totals
    torch.cuda.synchronize()                # and waits here for the copy and paste launches
    if it >= 3:
        ts.append((time.perf_counter() - t0) * 1e6)
call_us = float(np.median(ts))

from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(20):
        flush.zero_()
        step()
    torch.cuda.synchronize()
kus = {}
for ev in prof.key_averages():
    for key in KERNELS:
        if key in ev.key and ev.count:
            kus[key] = kus.get(key, 0.0) + ev.self_device_time_total / 20      # us per call

torch.set_num_threads(1)
host = []
for it in range(3):
    t0 = time.perf_counter()
    for f, g, gn, m, mn, a in zip(frames, gt, gt_names, inst, inst_names, angles):
        RP.rotate_paste_frame(f, f, g, gn, m, mn, a)
    host.append((time.perf_counter() - t0) * 1e3)

card = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                       "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
tiles = sum(-(-f.shape[0] // 1024) for f in frames)
member_mb = (4.0 * stride * n_in + 40 * tiles * (128 + 4)) / 1e6       # rows read; ballot words + tile counts written
move_mb = (4.0 * stride * n_in + 4.0 * stride * n_out) / 1e6            # destination rows read, output rows written
move_us = kus.get("rp_copy_dst_kernel", 0) + kus.get("rp_paste_kernel", 0)


def rate(mb, us):
    return (f"{mb / us * 1e3:.0f} GB/s, {100 * mb / us * 1e3 / peak:.1f}% of {peak:.0f} GB/s" if us else "not measured")


lines = [
    "# Rotate-paste on the device (K0 rotate-paste kernels)",
    "",
    f"Card: {card} (name, power limit), read in the same run.  `scripts/bench_rotate_paste.py`: four nus_0075 frames "
    f"({n_in} points, stride {stride}, collated), each its own source; 40 destination boxes and 40 instance boxes per "
    f"frame, 3 PolarMix angles ({4 * 3 * 40} candidates, {acc} accepted), {n_out} points out.  Kernel times: "
    "torch.profiler, mean of 20 calls; L2 flushed before each call.",
    "",
    "| launch | us per call |",
    "|---|---|",
]
for key in KERNELS:
    lines.append(f"| {key} | {kus.get(key, float('nan')):.1f} |")
lines += [
    f"| whole call (rotate_paste_points: host candidates and tables, upload, 5 launches, flags back; host clock, median "
    f"of 20) | {call_us:.1f} |",
    "",
    f"Membership pass (rp_member_kernel): {member_mb:.1f} MB of algorithmic traffic (4*stride*N read, 132 bytes of words "
    f"and counts per box and tile written) = {rate(member_mb, kus.get('rp_member_kernel', 0))}.",
    "",
    f"Copy and paste (rp_copy_dst + rp_paste): {move_us:.1f} us for {move_mb:.1f} MB (4*stride*N read + 4*stride*N' "
    f"written) = {rate(move_mb, move_us)}.",
    "",
    f"Host: the restatement (tests/rotate_paste_oracle.py, numpy plus the C box ops of tests/gt_sampling_box_ops.c, one "
    f"thread) of the same four frames: {float(np.median(host)):.1f} ms (median of 3).  This is the restatement, not "
    "TODA's code.",
    "",
]
text = "\n".join(lines)
print(text)
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
open(args.out, "w").write(text)
