"""K0 timing on the bench batch: toda_points_select and the world transform.  CUDA events, L2 flushed between
iterations; prints the card's name and power limit and a markdown table (committed as profiles/r01_points_select.md and
profiles/r03_points_world_transform.md)."""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from tests import world_aug_oracle as WA
from toda_b200 import ops, synth
from toda_b200.pcdet_plugin.augmentor import DataAugmentor

dev = torch.device("cuda", 0)
frames, collated = synth.make_batch("nus_0075", 4)
offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(dev)
pts = torch.from_numpy(collated).to(dev)
raw = torch.from_numpy(np.concatenate(frames)).to(dev)
peak = 6545.6
if os.path.exists("MEASURED_PEAKS.json"):
    peak = json.load(open("MEASURED_PEAKS.json"))["hbm_gbs"]
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
r = synth.CONFIGS["nus_0075"]["pc_range"]
cases = [
    ("range mask (keeps all: frames are pre-masked)", pts, offs, ops.SELECT_RANGE_XY, [r[0], r[1], r[3], r[4]], False, False, 1),
    ("range mask, half range", pts, offs, ops.SELECT_RANGE_XY, [r[0] / 2, r[1] / 2, r[3] / 2, r[4] / 2], False, False, 1),
    ("collate (raw frames -> [b,x,y,z,..])", raw, offs, ops.SELECT_RANGE_XY, [-1e30, -1e30, 1e30, 1e30], False, True, 0),
    ("cutmix rectangle, inside", pts, None, ops.SELECT_RECT_XY, [-20.0, -30.0, 35.0, 25.0], False, False, 1),
    ("PolarMix sector, complement", pts, None, ops.SELECT_SECTOR, [0.3, 0.3 + 1.570796], True, False, 1),
]


def time_us(call):
    """Median of 9 timed calls after 3 warm-up calls, in microseconds; returns (us, result of the last call)."""
    ts = []
    for it in range(12):
        flush.zero_()
        torch.cuda._sleep(2000000)     # ~1 ms of GPU spin so that the host has queued the call before e0 is reached
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = call()
        e1.record()
        torch.cuda.synchronize()
        if it >= 3:
            ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), res


def row(name, n_in, n_out, us, mb):
    gbs = mb / us * 1e3
    print("| %s | %d | %d | %.1f | %.1f | %.0f | %.1f%% |" % (name, n_in, n_out, us, mb, gbs, 100 * gbs / peak))


card = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit",
                       "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("card: %s (name, power limit)" % card)
print()
print("| case | points in | points out | us | algorithmic MB | GB/s | share of HBM peak (%.0f GB/s) |" % peak)
print("|---|---|---|---|---|---|---|")
for name, p, o, mode, params, inv, addb, xc in cases:
    us, (out, oo) = time_us(lambda: ops.points_select(p, o, mode, params, invert=inv, add_batch_col=addb, x_col=xc, trim=False))
    kept = int(oo[-1].item())
    row(name, p.shape[0], kept, us, (4.0 * p.shape[1] * p.shape[0] + 4.0 * out.shape[1] * kept) / 1e6)

# world augmentations: flip x and y, rotation and scaling all active in every frame; each frame has its own draws
steps = [dict(NAME="random_world_flip", ALONG_AXIS_LIST=["x", "y"]),
         dict(NAME="random_world_rotation", WORLD_ROT_ANGLE=[-0.78539816, 0.78539816]),
         dict(NAME="random_world_scaling", WORLD_SCALE_RANGE=[0.95, 1.05])]
draws = [[[True, True], -0.6 + 0.4 * b, 0.97 + 0.02 * b] for b in range(len(frames))]
aug = DataAugmentor(steps)
world_ops = [op for s, st in enumerate(aug.data_augmentor_queue) for op in st.point_ops([d[s] for d in draws])]
for name, p, xc in [("world transform (flip x, flip y, rotate, scale), collated", pts, 1),
                    ("world transform (flip x, flip y, rotate, scale), raw frames", raw, 0)]:
    us, _ = time_us(lambda: ops.points_world_transform(p, offs, world_ops, x_col=xc))
    row(name, p.shape[0], p.shape[0], us, 2 * 4.0 * p.shape[1] * p.shape[0] / 1e6)

# the same augmentation of the same four frames as the reference runs it (the oracle's restatement, numpy and torch on
# one host thread per frame): CPU work that the device transform takes off the DataLoader workers
torch.set_num_threads(1)
host = []
for it in range(5):
    t0 = time.perf_counter()
    for f, d in zip(frames, draws):
        WA.world_augment(f, np.zeros((0, 7), np.float32), steps, d)
    host.append((time.perf_counter() - t0) * 1e3)
print()
print("host (CPU, one thread): the reference's world augmentations of the same %d frames: %.2f ms (median of 5)"
      % (len(frames), float(np.median(host))))
