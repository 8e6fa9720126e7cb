"""Generates tests/golden/points.npz: outputs of the REFERENCE'S OWN point pre-steps and mixers on small seeded inputs.

Run with a reference checkout:   TODA_REFERENCE=<rasd3/TODA clone> python tests/golden/make_golden_points.py
Functions driven (loaded by path from that checkout, oracle/reference_loader.py):
  * common_utils.mask_points_by_range + DataProcessor.mask_points_and_boxes_outside_range / shuffle_points
    (pcdet/utils/common_utils.py L60-63, pcdet/datasets/processor/data_processor.py L78-103)
  * inter_domain_point_cutmix (inter_domain_point_cutmix.py L10-90): points output; the crop rectangle it drew is
    recovered by recording its np.random draws
  * swap (inter_domain_point_polarmix.py L44-99, inc_method='center', use_pitch=False): points output
  * intra_domain_point_mixup (intra_domain_point_mixup.py L15-30): points output; lambda and both permutations recorded
  * DatasetTemplate.collate_batch's 'points' branch is three lines of numpy (dataset.py L173-178) and is restated in
    the fixture directly (the class cannot be imported: pcdet/datasets/__init__.py is a SyntaxError).
The fixtures are small (a few thousand points) and are what travels to the GPU box.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import reference_loader as R          # noqa: E402
from oracle import spconv_oracle as S             # noqa: E402
from toda_b200 import synth                       # noqa: E402

SEED = 666


class RandomLog:
    """Records np.random draws made by a reference function (so that the GPU path can be given the same decisions)."""

    def __init__(self):
        self.log = []
        self._orig = {}

    def __enter__(self):
        for name in ("rand", "choice", "permutation", "beta", "random"):
            orig = getattr(np.random, name)
            self._orig[name] = orig

            def wrapped(*a, _orig=orig, _name=name, **k):
                v = _orig(*a, **k)
                self.log.append((_name, np.array(v, copy=True)))
                return v
            setattr(np.random, name, wrapped)
        return self

    def __exit__(self, *exc):
        for name, orig in self._orig.items():
            setattr(np.random, name, orig)
        return False

    def all(self, name):
        return [v for n, v in self.log if n == name]


def small_frame(config, idx, n, window=None):
    pts = synth.make_frame(config, idx, shuffle=False)
    if window is not None:
        m = (np.abs(pts[:, 0]) < window) & (np.abs(pts[:, 1]) < window)
        pts = pts[m]
    step = max(1, pts.shape[0] // n)
    return np.ascontiguousarray(pts[::step][:n])


def main():
    ns = R.load(S.make_modules())
    ns.load_mixers()
    out = {}

    # ---- a-0 / a-0b: range mask + shuffle through the reference's DataProcessor
    pcr = np.array([-20.0, -12.0, -5.0, 20.0, 12.0, 3.0], dtype=np.float32)
    pts = small_frame("nus_0075", 3, 6000, window=30.0)
    # points exactly on the boundary (inclusive on both ends) and a NaN row
    edge = pts[:6].copy()
    edge[0, 0], edge[1, 0], edge[2, 1], edge[3, 1] = pcr[0], pcr[3], pcr[1], pcr[4]
    edge[4, 0] = np.nextafter(pcr[3], np.float32(np.inf))
    edge[5, 0] = np.nan
    pts = np.concatenate([pts, edge]).astype(np.float32)
    C = R.Cfg
    cfgs = [C(NAME="mask_points_and_boxes_outside_range", REMOVE_OUTSIDE_BOXES=True),
            C(NAME="shuffle_points", SHUFFLE_ENABLED=C(train=True, test=True))]
    np.random.seed(SEED)
    dp = ns.DataProcessor(cfgs, point_cloud_range=pcr, training=True, num_point_features=pts.shape[1])
    with RandomLog() as rl:
        dd = dp.forward(data_dict={"points": pts.copy()})
    mask = ns.common_utils.mask_points_by_range(pts, pcr)
    out["mask/points"], out["mask/pc_range"], out["mask/mask"] = pts, pcr, mask
    out["mask/shuffle_idx"] = rl.all("permutation")[0]
    out["mask/result"] = dd["points"]
    print("mask+shuffle:", pts.shape, "->", dd["points"].shape)

    # ---- f-1: cutmix rectangle (source = Waymo-shaped, target = nuScenes-shaped, as the reference asserts)
    src = small_frame("waymo_010", 1, 10000)[:, :5]
    tgt = small_frame("nus_0075", 2, 30000)[:, :5]
    pc_range = np.array([-54.0, -54.0, -5.0, 54.0, 54.0, 4.8])
    empty_boxes = np.zeros((0, 8), dtype=np.float32)
    np.random.seed(SEED + 1)
    with RandomLog() as rl:
        mixed = ns.cutmix.inter_domain_point_cutmix({"points": src.copy(), "gt_boxes": empty_boxes.copy()},
                                                    {"points": tgt.copy(), "gt_boxes": empty_boxes.copy()}, pc_range, "center")
    crop_range = 0.5 + rl.all("rand")[-1] * 0.5           # the accepted aspect draw is the last rand(2) (L29-36)
    centre_idx = int(rl.all("choice")[-1])                # the accepted centre is the last choice
    new_range = (pc_range[3:5] - pc_range[0:2]) * crop_range / 2.0
    centre = src[centre_idx, 0:3]
    out["cutmix/source"], out["cutmix/target"] = src, tgt
    out["cutmix/min_xy"], out["cutmix/max_xy"] = centre[:2] - new_range, centre[:2] + new_range
    out["cutmix/result"] = mixed["points"].astype(np.float32)
    print("cutmix:", src.shape, tgt.shape, "->", mixed["points"].shape, "rect", out["cutmix/min_xy"], out["cutmix/max_xy"])

    # ---- f-1: PolarMix sector swap (points part; no boxes)
    p1 = small_frame("waymo_010", 2, 8000)[:, :5]
    p2 = small_frame("nus_0075", 4, 8000)[:, :5]
    boxes = np.zeros((0, 8), dtype=np.float32)
    sectors = [(-2.0, -2.0 + 1.570796), (1.9, np.pi)]
    for j, (a0, a1) in enumerate(sectors):
        res, _ = ns.polarmix.swap(p1.copy(), p2.copy(), a0, a1, boxes.copy(), boxes.copy(), inc_method="center", use_pitch=False)
        out[f"polar{j}/pt1"], out[f"polar{j}/pt2"] = p1, p2
        out[f"polar{j}/angles"] = np.array([a0, a1], dtype=np.float64)
        out[f"polar{j}/result"] = res.astype(np.float32)
        print("polar swap", j, "->", res.shape)

    # ---- f-1: intra-domain mixup (prefixes of two shuffled frames)
    m1 = small_frame("nus_0075", 5, 5000)[:, :5]
    m2 = small_frame("nus_0075", 6, 4000)[:, :5]
    np.random.seed(SEED + 2)
    with RandomLog() as rl:
        mixed = ns.mixup.intra_domain_point_mixup({"points": m1.copy(), "gt_boxes": boxes.copy()},
                                                  {"points": m2.copy(), "gt_boxes": boxes.copy()}, alpha=2)
    perms = rl.all("permutation")
    out["mixup/points_1"], out["mixup/points_2"] = m1, m2
    out["mixup/lam"] = np.array(float(rl.all("beta")[0]))
    out["mixup/shuffle_idx_1"], out["mixup/shuffle_idx_2"] = perms[0], perms[1]
    out["mixup/result"] = mixed["points"].astype(np.float32)
    print("mixup:", m1.shape, m2.shape, "lam", out["mixup/lam"], "->", mixed["points"].shape)

    # ---- f-1 (box side, first piece): get_points_in_box, pure numpy in the reference (augmentor_utils.py L474-491)
    bp = small_frame("nus_0075", 9, 6000, window=25.0)[:, :5]
    rngb = np.random.default_rng(SEED + 3)
    centres = bp[rngb.integers(0, bp.shape[0], 6), :3]
    boxes_pb = np.concatenate([centres, rngb.uniform([1.5, 1.0, 1.0], [8.0, 4.0, 3.0], (6, 3)), rngb.uniform(-np.pi, np.pi, (6, 1)),
                               np.ones((6, 1))], axis=1).astype(np.float32)
    masks = np.stack([ns.augmentor_utils.get_points_in_box(bp, b)[1] for b in boxes_pb])
    out["inbox/points"], out["inbox/boxes"], out["inbox/masks"] = bp, boxes_pb, masks
    print("points in boxes:", bp.shape, "boxes", boxes_pb.shape, "inside counts", masks.sum(1))

    # ---- a-2: collate (three numpy lines of dataset.py L173-178, restated; see the module docstring)
    frames = [small_frame("nus_0075", 7 + i, 700 + 100 * i) for i in range(3)]
    collated = np.concatenate([np.pad(f, ((0, 0), (1, 0)), mode="constant", constant_values=i) for i, f in enumerate(frames)], axis=0)
    for i, f in enumerate(frames):
        out[f"collate/frame{i}"] = f
    out["collate/result"] = collated

    np.savez_compressed(os.path.join(HERE, "points.npz"), **out)
    print("wrote", os.path.join(HERE, "points.npz"), os.path.getsize(os.path.join(HERE, "points.npz")) // 1024, "KB")


if __name__ == "__main__":
    main()
