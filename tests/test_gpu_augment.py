"""World augmentations on the GPU (K0 world transform, pcdet_plugin.augmentor.DataAugmentor) against the restatement of
OpenPCDet v0.5.2's DataAugmentor in tests/world_aug_oracle.py, with the same recorded draws.  Points must be bit-identical
(signed zeros included, NaN compared as NaN); boxes must be equal in their own dtype."""
import itertools

import numpy as np
import pytest
import torch

from oracle import points as OP
from tests import parity_utils as PU
from tests import world_aug_oracle as WA

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32 = np.float32
FLIP = PU.Cfg(NAME="random_world_flip", ALONG_AXIS_LIST=["x", "y"])
ROT = PU.Cfg(NAME="random_world_rotation", WORLD_ROT_ANGLE=[-0.78539816, 0.78539816])
SCALE = PU.Cfg(NAME="random_world_scaling", WORLD_SCALE_RANGE=[0.95, 1.05])
SCALE_OFF = PU.Cfg(NAME="random_world_scaling", WORLD_SCALE_RANGE=[1.0, 1.0005])     # narrower than 1e-3: no draw, no step


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(((a.view(np.int32) == b.view(np.int32)) | (np.isnan(a) & np.isnan(b))).all())


def _special_frame(n):
    """Rows built from 0, -0, +-inf, NaN, a denormal and ordinary values in x, y, z."""
    vals = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, 1.5, -37.25], F32)
    xyz = np.array(list(itertools.product(vals, repeat=3)), F32)[:n]
    return np.concatenate([xyz, np.tile(np.array([[0.25, -0.0]], F32), (xyz.shape[0], 1))], 1)


def _frames():
    """Four full-size frames, plus an empty frame, a 1-point frame, the two frames on either side of torch's dispatch
    (44 and 45 rows) and frames of special values on both sides of it."""
    from toda_b200 import synth
    full = [synth.make_frame("nus_0075", i) for i in range(4)]
    rng = np.random.default_rng(9)
    small = [(rng.standard_normal((n, 5)) * 30).astype(F32) for n in (1, 44, 45)]
    return [full[0], full[1][:0], small[0], full[1], small[1], small[2], full[2], _special_frame(44), _special_frame(512),
            full[3]]


def _collate(frames, x_col):
    raw = np.concatenate(frames)
    pts = OP.collate_points(frames).astype(F32) if x_col == 1 else raw
    offs = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)
    return pts, offs


ORDERS = [[FLIP, ROT, SCALE], [SCALE, ROT, FLIP], [ROT, FLIP, SCALE], [FLIP, ROT, SCALE_OFF],
          [PU.Cfg(NAME="random_world_flip", ALONG_AXIS_LIST=["y", "x"]), SCALE, PU.Cfg(NAME="random_world_rotation", WORLD_ROT_ANGLE=0.4)]]


@pytest.mark.parametrize("x_col", [0, 1])
@pytest.mark.parametrize("order", range(len(ORDERS)))
def test_points_bit_identical_to_the_reference(order, x_col):
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    steps = ORDERS[order]
    frames = _frames()
    pts, offs = _collate(frames, x_col)
    aug = DataAugmentor(steps, x_col=x_col)
    np.random.seed(100 + order)
    dd = aug.forward({"points": _t(pts), "point_frame_offsets": _t(offs)})
    draws = dd["world_aug_draws"]
    assert len(draws) == len(frames)
    np.random.seed(100 + order)
    assert [WA.draw_world_augmentations(steps) for _ in frames] == draws       # frame by frame, config order
    if steps[-1] is SCALE_OFF:
        assert all(d[-1] is None for d in draws)
    got = dd["points"].cpu().numpy()
    want = [WA.world_augment(f, np.zeros((0, 7), F32), steps, d)[0] for f, d in zip(frames, draws)]
    want = OP.collate_points(want).astype(F32) if x_col == 1 else np.concatenate(want)
    assert got.shape == want.shape
    for b in range(len(frames)):
        lo, hi = offs[b], offs[b + 1]
        assert _bits_equal(got[lo:hi], want[lo:hi]), f"frame {b} ({hi - lo} rows) differs"
    # replaying the recorded draws gives the same points
    again = aug.forward({"points": _t(pts), "point_frame_offsets": _t(offs), "world_aug_draws": draws})
    assert _bits_equal(again["points"].cpu().numpy(), got)


def test_one_frame_without_offsets_and_empty_input():
    from toda_b200 import ops
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    rng = np.random.default_rng(3)
    for n in (0, 44, 45, 1000):
        p = (rng.standard_normal((n, 4)) * 20).astype(F32)
        np.random.seed(n)
        dd = DataAugmentor([FLIP, ROT, SCALE], x_col=0).forward({"points": _t(p)})
        want, _ = WA.world_augment(p, np.zeros((0, 7), F32), [FLIP, ROT, SCALE], dd["world_aug_draws"][0])
        assert _bits_equal(dd["points"].cpu().numpy(), want)
    p = _t(rng.standard_normal((10, 4)).astype(F32))
    assert torch.equal(ops.points_world_transform(p, None, []), p)


@pytest.mark.parametrize("cols", [7, 9, 10])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_gt_boxes_match_the_reference(cols, dtype):
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    steps = [FLIP, ROT, SCALE]
    rng = np.random.default_rng(cols)
    frames = [(rng.standard_normal((n, 5)) * 20).astype(F32) for n in (300, 0, 50)]
    boxes = [(rng.standard_normal((m, cols)) * 10).astype(dtype) for m in (12, 44, 45)]
    boxes[0][:, 6] = np.linspace(-7, 7, 12)                             # headings outside [-pi, pi) for limit_period
    mask = [np.arange(m) % 3 != 1 for m in (12, 44, 45)]
    names = [np.array(["car"] * m) for m in (12, 44, 45)]
    pts, offs = _collate(frames, 1)
    aug = DataAugmentor(steps)
    np.random.seed(cols)
    dd = aug.forward({"points": _t(pts), "point_frame_offsets": _t(offs), "gt_boxes": [b.copy() for b in boxes],
                      "gt_boxes_mask": mask, "gt_names": names})
    assert "gt_boxes_mask" not in dd
    for b in range(3):
        want_p, want_b = WA.world_augment(frames[b], boxes[b], steps, dd["world_aug_draws"][b])
        got_b = dd["gt_boxes"][b]
        assert got_b.dtype == dtype and np.array_equal(got_b, want_b[mask[b]]), b
        assert dd["gt_names"][b].shape[0] == mask[b].sum()
        assert _bits_equal(dd["points"][offs[b]:offs[b + 1], 1:].cpu().numpy(), want_p)
        assert np.all(got_b[:, 6] >= -np.pi - 1e-6) and np.all(got_b[:, 6] < np.pi + 1e-6)


def test_augmentor_then_preprocessor_then_voxelizer():
    """DataAugmentor -> PointPreprocessor (range mask, shuffle with a given index) -> MeanVFE.voxelize equals the oracle
    voxelizer run on the oracle's augmented, masked and shuffled frames."""
    import toda_b200.pcdet_plugin as P
    from toda_b200 import synth
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    from toda_b200.pcdet_plugin.processor import PointPreprocessor
    cfg = synth.CONFIGS["nus_0075"]
    pcr = cfg["pc_range"]
    steps = [FLIP, ROT, SCALE]
    frames = [synth.make_frame("nus_0075", i) for i in range(3)]
    frames.insert(1, (np.random.default_rng(1).standard_normal((44, 5)) * 20).astype(F32))
    pts, offs = _collate(frames, 1)
    np.random.seed(77)
    draws = [WA.draw_world_augmentations(steps) for _ in frames]
    want = [OP.mask_points_outside_range(WA.world_augment(f, np.zeros((0, 7), F32), steps, d)[0], pcr) for f, d in zip(frames, draws)]
    rng = np.random.default_rng(5)
    perms = [rng.permutation(w.shape[0]) for w in want]
    starts = np.cumsum([0] + [w.shape[0] for w in want])
    shuffle_idx = np.concatenate([p + s for p, s in zip(perms, starts)]).astype(np.int32)
    want = [OP.shuffle_points(w, p) for w, p in zip(want, perms)]

    aug = DataAugmentor(steps)
    pp = PointPreprocessor([PU.Cfg(NAME="mask_points_and_boxes_outside_range", REMOVE_OUTSIDE_BOXES=True),
                            PU.Cfg(NAME="shuffle_points", SHUFFLE_ENABLED=PU.Cfg(train=True, test=True)),
                            PU.Cfg(NAME="transform_points_to_voxels_placeholder", VOXEL_SIZE=cfg["voxel_size"])],
                           pcr, training=True, num_point_features=5)
    vfe = P.MeanVFE(PU.Cfg(MAX_POINTS_PER_VOXEL=cfg["max_points"], MAX_NUMBER_OF_VOXELS=cfg["max_voxels"]), 5,
                    voxel_size=cfg["voxel_size"], point_cloud_range=pcr, grid_size=pp.grid_size).to(DEV).train()
    bd = pp.forward(aug.forward({"points": _t(pts), "point_frame_offsets": _t(offs), "world_aug_draws": draws,
                                 "shuffle_idx": shuffle_idx, "batch_size": len(frames)}))
    assert _bits_equal(bd["points"].cpu().numpy(), OP.collate_points(want).astype(F32))
    bd = vfe.voxelize(bd)
    coords = bd["voxel_coords"].cpu().numpy()
    counts = np.bincount(coords[:, 0], minlength=len(frames)).tolist()
    got = (bd["voxels"].cpu().numpy(), coords, bd["voxel_num_points"].cpu().numpy(), np.array(counts + [sum(counts)]))
    ref = PU.oracle_voxelize_batch(want, pcr, cfg["voxel_size"], cfg["max_points"], cfg["max_voxels"]["train"])
    PU.assert_voxels_equal(got, ref, exact_order=False)


def test_argument_errors():
    from toda_b200 import ops
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    p = _t(np.zeros((10, 4), F32))
    offs = _t(np.array([0, 4, 10], np.int32))
    with pytest.raises(ValueError, match="stride"):
        ops.points_world_transform(p, offs, [], x_col=2)                   # x, y, z do not fit
    with pytest.raises(ValueError, match="at most 4"):
        ops.points_world_transform(p, offs, [(ops.WORLD_SCALE, [1.0, 1.0])] * 5)
    with pytest.raises(ValueError, match="kind"):
        ops.points_world_transform(p, offs, [(7, [1.0, 1.0])])
    with pytest.raises(ValueError, match="value"):
        ops.points_world_transform(p, offs, [(ops.WORLD_ROTATE, [1.0, 0.0])])   # one (cos, sin) for two frames
    with pytest.raises(ValueError, match="batch"):
        ops.points_world_transform(_t(np.zeros((70, 4), F32)), _t(np.arange(66, dtype=np.int32)), [])
    L = ops._C.lib()
    assert L.toda_points_world_transform(None, 10, 4, 2, None, 1, 0, None, None, None, None) == -1
    assert b"layout" in L.toda_last_error()
    kinds, prm = ops._C.ints([9]), ops._C.floats([0.0, 0.0])
    assert L.toda_points_world_transform(None, 0, 4, 0, None, 1, 1, kinds, prm, None, None) == -1
    assert b"kind" in L.toda_last_error()
    assert L.toda_points_world_transform(None, 5, 4, 0, None, 1, 0, None, None, None, None) == -1
    assert b"null" in L.toda_last_error()
    aug = DataAugmentor([FLIP, ROT])
    with pytest.raises(ValueError, match="list of per-frame"):
        aug.forward({"points": p, "point_frame_offsets": offs, "gt_boxes": np.zeros((2, 5, 7), F32)})
    with pytest.raises(NotImplementedError, match="random_local_scaling"):
        DataAugmentor([FLIP, PU.Cfg(NAME="random_local_scaling", LOCAL_SCALE_RANGE=[0.95, 1.05])])
    with pytest.raises(NotImplementedError, match="gt_sampling"):
        DataAugmentor([PU.Cfg(NAME="gt_sampling"), FLIP])
    assert len(DataAugmentor([PU.Cfg(NAME="gt_sampling"), FLIP], host_steps=["gt_sampling"]).data_augmentor_queue) == 1


def test_pipeline_preprocess_equals_inline_steps():
    """InputPipeline(preprocess=...) runs the augmentation and the point pre-steps on its side stream: results are
    bit-identical to the same steps run in-line before the VFE (fp32)."""
    from tests.test_gpu_pipeline import _batches, _modules, _run
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    from toda_b200.pcdet_plugin.processor import PointPreprocessor
    from toda_b200.pipeline import InputPipeline
    dev = torch.device("cuda", 0)
    vfe, net, hc, pcr = _modules(dev, "fp32")
    aug = DataAugmentor([FLIP, ROT, SCALE])
    pp = PointPreprocessor([PU.Cfg(NAME="mask_points_and_boxes_outside_range")], pcr, training=True, num_point_features=5)
    host = _batches(pcr, 3)
    np.random.seed(21)
    draws = [[WA.draw_world_augmentations([FLIP, ROT, SCALE]) for _ in range(2)] for _ in host]
    state = {k: v.clone() for k, v in net.state_dict().items()}
    want = []
    for (p, o), d in zip(host, draws):
        bd = pp.forward(aug.forward({"points": p.to(dev), "point_frame_offsets": o.to(dev), "batch_size": 2, "world_aug_draws": d}))
        want.append(_run(net, hc, vfe(bd)))
    net.load_state_dict(state)
    pipe = InputPipeline(vfe, net, dev, reserve_bytes=64 << 20, preprocess=lambda bd: pp.forward(aug.forward(bd)))
    pinned = [(p.pin_memory(), o.pin_memory()) for p, o in host]

    def submit(i):
        return pipe.submit({"points": pinned[i][0], "point_frame_offsets": pinned[i][1], "batch_size": 2, "world_aug_draws": draws[i]})
    h = submit(0)
    for i in range(3):
        bd = pipe.consume(h)
        if i + 1 < 3:
            h = submit(i + 1)
        got = _run(net, hc, bd)
        sf_w, idx_w, g_w = want[i]
        assert torch.equal(got[1], idx_w) and torch.equal(got[0], sf_w)
        for name in g_w:
            assert torch.equal(got[2][name], g_w[name]), name
    torch.cuda.synchronize()
