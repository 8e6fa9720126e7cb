"""Generates the committed golden fixtures in tests/golden/*.npz.

Run with a reference checkout:   TODA_REFERENCE=<rasd3/TODA clone> python tests/golden/make_golden.py
It drives the REFERENCE'S OWN files of that checkout (data_processor.py, mean_vfe.py,
spconv_backbone.py, height_compression.py -- loaded by path, oracle/reference_loader.py) with the
CPU oracle standing in for the absent third-party `spconv`/`cumm` packages, on small seeded inputs,
and records inputs + outputs.  The GPU parity tests replay the inputs through the CUDA path and
compare.  The reference is not part of this repository; the fixtures are what travels.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import reference_loader as R          # noqa: E402
from oracle import spconv_oracle as S             # noqa: E402
from toda_b200 import synth                       # noqa: E402

SEED = 666   # the reference's --fix_random_seed value (pcdet/utils/common_utils.py L102-107)


def processor_cfgs(voxel_size, max_points, max_voxels):
    C = R.Cfg
    return [
        C(NAME="mask_points_and_boxes_outside_range", REMOVE_OUTSIDE_BOXES=True),
        C(NAME="shuffle_points", SHUFFLE_ENABLED=C(train=True, test=True)),
        C(NAME="transform_points_to_voxels", VOXEL_SIZE=voxel_size, MAX_POINTS_PER_VOXEL=max_points,
          MAX_NUMBER_OF_VOXELS=C(train=max_voxels, test=max_voxels)),
    ]


class Recorder:
    """Wraps shuffle_points so that the exact point order fed to the voxelizer is captured."""

    def __init__(self, dp):
        self.points = None
        inner = dp.data_processor_queue[-1]

        def spy(data_dict):
            self.points = data_dict["points"].copy()
            return inner(data_dict=data_dict)
        dp.data_processor_queue[-1] = spy


def golden_voxelize(ns):
    cases = {}
    base = synth.make_frame("nus_0075", 0, shuffle=False)
    waymo = synth.make_frame("waymo_010", 0, shuffle=False)
    specs = [
        # name, points, range, voxel, K, max_voxels
        ("crop_nus", base, [4.0, -2.4, -5.0, 8.8, 2.4, 3.0], [0.075, 0.075, 0.2], 10, 20000),
        ("crop_nus_capped", base, [4.0, -2.4, -5.0, 8.8, 2.4, 3.0], [0.075, 0.075, 0.2], 3, 700),
        ("crop_waymo", waymo[::2], [5.0, -6.4, -2.0, 17.8, 6.4, 4.0], [0.1, 0.1, 0.15], 5, 150000),
        ("coarse_full_nus", base[::7], [-51.2, -51.2, -5.0, 51.2, 51.2, 3.0], [0.8, 0.8, 0.4], 4, 3000),
    ]
    for name, pts, rng_, vs, k, mv in specs:
        pcr = np.array(rng_, dtype=np.float32)
        # the mask step keeps x/y in range; pre-crop generously so that fixtures stay small but
        # still contain out-of-range points (z and the far side) for the voxelizer to reject
        m = (pts[:, 0] > rng_[0] - 0.5) & (pts[:, 0] < rng_[3] + 0.5) & (pts[:, 1] > rng_[1] - 0.5) & (pts[:, 1] < rng_[4] + 0.5)
        raw = np.ascontiguousarray(pts[m])
        np.random.seed(SEED)
        dp = ns.DataProcessor(processor_cfgs(vs, k, mv), point_cloud_range=pcr, training=True,
                              num_point_features=raw.shape[1])
        rec = Recorder(dp)
        dd = dp.forward(data_dict={"points": raw.copy(), "use_lead_xyz": True})
        vfe = ns.MeanVFE(R.Cfg(), raw.shape[1])
        bd = vfe({"voxels": torch.from_numpy(dd["voxels"]), "voxel_num_points": torch.from_numpy(dd["voxel_num_points"]).float()})
        cases[name] = dict(points=rec.points, pc_range=pcr, voxel_size=np.array(vs, np.float32),
                           grid_size=dp.grid_size, max_points=k, max_voxels=mv, voxels=dd["voxels"],
                           voxel_coords=dd["voxel_coords"], voxel_num_points=dd["voxel_num_points"],
                           voxel_features=bd["voxel_features"].numpy())
        print(name, raw.shape, "->", rec.points.shape, "voxels", dd["voxels"].shape, "grid", dp.grid_size)
    flat = {f"{c}/{k}": np.asarray(v) for c, d in cases.items() for k, v in d.items()}
    np.savez_compressed(os.path.join(HERE, "voxelize.npz"), **flat)


def collate(samples):
    """pcdet/datasets/dataset.py L171-178 for the three voxel keys."""
    voxels = np.concatenate([s[0] for s in samples])
    num = np.concatenate([s[2] for s in samples])
    coords = np.concatenate([np.pad(s[1], ((0, 0), (1, 0)), mode="constant", constant_values=i)
                             for i, s in enumerate(samples)])
    return voxels, coords, num


def stage2_frames(f):
    """Two samples shaped like a TODA stage-2 batch (BASELINE configs[3]): an intra-domain mixup of two single-sweep
    nuScenes-shaped frames (intra_domain_point_mixup.py L23-27, lam = 0.6) and a polar-sector swap of a Waymo-shaped frame
    into a nuScenes-shaped one (inter_domain_point_polarmix.py L72-95, pi/2 sector).  The mixers themselves are pinned by
    tests/golden/points.npz; here they only build the inputs, which are stored in the fixture."""
    from oracle import points as OP
    a, b = synth.make_frame("toda_stage2", 0)[:, :f], synth.make_frame("toda_stage2", 1)[:, :f]
    rng = np.random.default_rng(4004)
    mix = OP.mixup_points(a, b, 0.6, rng.permutation(a.shape[0]), rng.permutation(b.shape[0]))
    w = synth.make_frame("waymo_010", 0)[:, :f]
    swap = OP.polar_swap_points(synth.make_frame("toda_stage2", 2)[:, :f], w, 0.3, 0.3 + np.pi / 2)
    return [np.ascontiguousarray(mix), np.ascontiguousarray(swap)]


def golden_backbone(ns, cls_name, fname, frame_cfg, crop, vs, k, f):
    pcr = np.array(crop, dtype=np.float32)
    samples = []
    frames = stage2_frames(f) if frame_cfg == "toda_stage2" else None
    for fi in range(2):
        pts = frames[fi] if frames is not None else synth.make_frame(frame_cfg, fi, shuffle=True)[:, :f]
        np.random.seed(SEED + fi)
        dp = ns.DataProcessor(processor_cfgs(vs, k, 4000), point_cloud_range=pcr, training=True, num_point_features=f)
        dd = dp.forward(data_dict={"points": np.ascontiguousarray(pts), "use_lead_xyz": True})
        samples.append((dd["voxels"], dd["voxel_coords"], dd["voxel_num_points"]))
        grid = dp.grid_size
    voxels, coords, num = collate(samples)
    # load_data_to_gpu (pcdet/models/__init__.py L34): everything becomes float32
    bd = {"voxels": torch.from_numpy(voxels).float(), "voxel_coords": torch.from_numpy(coords).float(),
          "voxel_num_points": torch.from_numpy(num).float(), "batch_size": 2}
    vfe = ns.MeanVFE(R.Cfg(), f)
    bd = vfe(bd)
    torch.manual_seed(SEED)
    net = getattr(ns, cls_name)(R.Cfg(), f, grid)
    hc = ns.HeightCompression(R.Cfg(NUM_BEV_FEATURES=net.num_point_features * 2))
    out = {}
    wsum = float(sum(p.detach().double().abs().sum() for p in net.parameters()))
    # ---- train-mode forward + backward (BatchNorm batch statistics) ----
    net.train()
    vf = bd["voxel_features"].clone().requires_grad_(True)
    b1 = hc(net({"voxel_features": vf, "voxel_coords": bd["voxel_coords"], "batch_size": 2}))
    sf = b1["spatial_features"]
    gen = torch.Generator().manual_seed(SEED)
    cot = torch.randn(sf.shape, generator=gen)
    loss = (sf * cot).sum()
    loss.backward()
    enc = b1["encoded_spconv_tensor"]
    out.update(train_enc_features=enc.features.detach().numpy(), train_enc_indices=enc.indices.numpy(),
               train_dvoxel_features=vf.grad.numpy(), train_loss=np.float64(loss.item()))
    for name, t in b1["multi_scale_3d_features"].items():
        out[f"train_{name}_features"] = t.features.detach().numpy()
        out[f"train_{name}_indices"] = t.indices.numpy()
    names, norms = [], []
    for n_, p in net.named_parameters():
        names.append(n_)
        norms.append(float(p.grad.double().norm()))
    out["grad_names"] = np.array(names)
    out["grad_norms"] = np.array(norms)
    out["grad_conv_input_weight"] = net.conv_input[0].weight.grad.numpy()
    out["grad_conv_out_weight"] = net.conv_out[0].weight.grad.numpy()
    out["running_mean_conv_input"] = net.conv_input[1].running_mean.numpy().copy()
    out["running_var_conv_input"] = net.conv_input[1].running_var.numpy().copy()
    # ---- eval-mode forward from a fresh copy of the same initial weights ----
    torch.manual_seed(SEED)
    net2 = getattr(ns, cls_name)(R.Cfg(), f, grid)
    net2.eval()
    with torch.no_grad():
        b2 = hc(net2({"voxel_features": bd["voxel_features"], "voxel_coords": bd["voxel_coords"], "batch_size": 2}))
    enc2 = b2["encoded_spconv_tensor"]
    out.update(eval_enc_features=enc2.features.numpy(), eval_enc_indices=enc2.indices.numpy(),
               eval_bev_sum=np.float64(b2["spatial_features"].double().sum().item()),
               bev_shape=np.array(b2["spatial_features"].shape))
    out.update(voxels=voxels, voxel_coords=coords, voxel_num_points=num, voxel_features=bd["voxel_features"].numpy(),
               grid_size=np.asarray(grid), weight_abs_sum=np.float64(wsum), seed=np.int64(SEED),
               pc_range=pcr, voxel_size=np.array(vs, np.float32))
    np.savez_compressed(os.path.join(HERE, fname), **out)
    print(cls_name, "voxels", voxels.shape, "enc", enc.features.shape, "bev", tuple(sf.shape), "loss", loss.item())


def main():
    from tests import parity_utils as PU
    torch.set_num_threads(PU.GOLDEN_THREADS)      # the replay in tests/test_plugin_topology.py runs at the same count
    ns = R.load(S.make_modules())
    if "--stage2" in sys.argv:
        # TODA stage-1/2 grid: z range -5 .. 4.8 -> 49 bins -> sparse_shape [50, ., .] (shape chain 50 -> 25 -> 13 -> 6 -> 2), F = 4
        # (tools/cfgs/stage2_advmix/centerpoint_5_lab_95_unlab_nus_frames_advmix.yaml L13-14, L56-80)
        golden_backbone(ns, "VoxelResBackBone8x", "backbone_res_stage2.npz", "toda_stage2",
                        [4.0, -4.8, -5.0, 13.6, 4.8, 4.8], [0.075, 0.075, 0.2], 10, 4)
        return
    golden_voxelize(ns)
    golden_backbone(ns, "VoxelResBackBone8x", "backbone_res.npz", "nus_0075",
                    [4.0, -2.4, -5.0, 8.8, 2.4, 3.0], [0.075, 0.075, 0.2], 10, 5)
    golden_backbone(ns, "VoxelBackBone8x", "backbone_voxel.npz", "waymo_010",
                    [5.0, -3.2, -2.0, 11.4, 3.2, 4.0], [0.1, 0.1, 0.15], 5, 5)


if __name__ == "__main__":
    main()
