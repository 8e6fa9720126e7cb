"""gt_sampling timing on the bench batch (four nus_0075 frames, nuScenes SAMPLE_GROUPS, 40 synthetic gt boxes per frame,
a synthetic database of 200 objects per class written to a temporary directory).  Kernel times from torch.profiler
(CUDA activity), the whole step from a host clock around a call that ends in a synchronise, the L2 flushed between
iterations; prints the card's name and power limit and writes a markdown table (committed as profiles/r05_gt_sampling.md).

    python scripts/bench_gt_sampling.py [--out PATH]
"""
import argparse, json, os, subprocess, sys, tempfile, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from tests import gt_sampling_oracle as GS
from tests import parity_utils as PU
from toda_b200 import synth
from toda_b200.pcdet_plugin.augmentor import DataAugmentor

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="profiles/r05_gt_sampling.md")
args = ap.parse_args()

CLASSES = ["car", "truck", "construction_vehicle", "bus", "trailer", "barrier", "motorcycle", "bicycle", "pedestrian",
           "traffic_cone"]
GROUPS = ["car:2", "truck:3", "construction_vehicle:7", "bus:4", "trailer:6", "barrier:2", "motorcycle:6", "bicycle:6",
          "pedestrian:2", "traffic_cone:2"]
dev = torch.device("cuda", 0)
peak = 7700.0
if os.path.exists("MEASURED_PEAKS.json"):
    peak = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"]
tmp = tempfile.mkdtemp()
info = GS.write_database(tmp, CLASSES, 200, 5, seed=1)
cfg = PU.Cfg(NAME="gt_sampling", DB_INFO_PATH=[info], PREPARE={"filter_by_min_points": [f"{c}:5" for c in CLASSES]},
             SAMPLE_GROUPS=GROUPS, NUM_POINT_FEATURES=5, REMOVE_EXTRA_WIDTH=[0.0, 0.0, 0.0], LIMIT_WHOLE_SCENE=False)
frames, collated = synth.make_batch("nus_0075", 4)
offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(dev)
pts = torch.from_numpy(collated).to(dev)
rng = np.random.default_rng(3)
gt_boxes, gt_names = [], []
for _ in frames:
    m = 40
    gt_boxes.append(np.concatenate([rng.uniform(-50, 50, (m, 2)), rng.uniform(-2, 0, (m, 1)), rng.uniform(0.5, 5, (m, 3)),
                                    rng.uniform(-np.pi, np.pi, (m, 1)), rng.normal(0, 2, (m, 2))], 1).astype(np.float32))
    gt_names.append(np.array([CLASSES[i] for i in rng.integers(0, 10, m)]))
aug = DataAugmentor([cfg], class_names=CLASSES, root_path=tmp)
np.random.seed(0)
draws = [[aug.data_augmentor_queue[0].draw(n)] for n in gt_names]


def step():
    return aug.forward({"points": pts, "point_frame_offsets": offs, "gt_boxes": gt_boxes, "gt_names": gt_names,
                        "world_aug_draws": draws})


flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
out = step()
n_in, n_out = pts.shape[0], out["points"].shape[0]
n_samples = sum(len(x) for d in draws for x in d[0])
acc = sum(b.shape[0] - g.shape[0] for b, g in zip(out["gt_boxes"], gt_boxes))
ts = []
for it in range(23):
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    step()                                  # ends in the device-to-host copy of the flags and offsets (a synchronise)
    if it >= 3:
        ts.append((time.perf_counter() - t0) * 1e6)
step_us = float(np.median(ts))

from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(20):
        flush.zero_()
        step()
    torch.cuda.synchronize()
kus = {}
for ev in prof.key_averages():
    for key in ("gts_accept_kernel", "select_flag_kernel", "select_copy_kernel", "gts_paste_kernel"):
        if key in ev.key and ev.count:
            kus[key] = kus.get(key, 0.0) + ev.self_device_time_total / 20      # us per batch (all launches of the batch)

torch.set_num_threads(1)
host = []
for it in range(3):
    ref = GS.DataBaseSampler(tmp, cfg, CLASSES)
    np.random.seed(0)
    t0 = time.perf_counter()
    for f, g, nm in zip(frames, gt_boxes, gt_names):
        ref({"points": f, "gt_boxes": g, "gt_names": nm, "gt_boxes_mask": np.ones(g.shape[0], bool)})
    host.append((time.perf_counter() - t0) * 1e3)

card = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                       "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
stride = pts.shape[1]
mb = (4.0 * stride * n_in + 4.0 * stride * n_out) / 1e6
move_us = kus.get("select_flag_kernel", 0) + kus.get("select_copy_kernel", 0) + kus.get("gts_paste_kernel", 0)
lines = [
    "# gt_sampling on the device (K0 gt_sampling kernels)",
    "",
    f"Card: {card} (name, power limit), read in the same run.  `scripts/bench_gt_sampling.py`: four nus_0075 frames "
    f"({n_in} points, stride {stride}), 40 gt boxes per frame, nuScenes SAMPLE_GROUPS ({n_samples} samples drawn, {acc} "
    f"accepted), {n_out} points out.  Kernel times: torch.profiler, mean of 20 batches; L2 flushed before each batch.",
    "",
    "| launch | us per batch |",
    "|---|---|",
]
for key in ("gts_accept_kernel", "select_flag_kernel", "select_copy_kernel", "gts_paste_kernel"):
    lines.append(f"| {key} | {kus.get(key, float('nan')):.1f} |")
lines += [
    f"| whole step (DataAugmentor.forward: host tables, upload, 4 launches, flags back; host clock, median of 20) | {step_us:.1f} |",
    "",
    f"Removal and paste pass (select_flag + select_copy + gts_paste): {move_us:.1f} us for {mb:.1f} MB of algorithmic traffic "
    f"(4*stride*N read + 4*stride*N' written) = {mb / move_us * 1e3 if move_us else float('nan'):.0f} GB/s, "
    f"{100 * mb / move_us * 1e3 / peak if move_us else float('nan'):.1f}% of {peak:.0f} GB/s.",
    "",
    f"Host: the restatement (tests/gt_sampling_oracle.py, numpy plus the C box ops, one thread) of the same four frames: "
    f"{float(np.median(host)):.1f} ms (median of 3).  This is the restatement, not pcdet itself.",
    "",
]
text = "\n".join(lines)
print(text)
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
open(args.out, "w").write(text)
