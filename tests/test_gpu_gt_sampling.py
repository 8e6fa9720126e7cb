"""gt_sampling on the GPU (K0 gt_sampling kernels, pcdet_plugin.augmentor.DataAugmentor with a device database) against
the restatement of OpenPCDet v0.5.2's DataBaseSampler in tests/gt_sampling_oracle.py, with the same np.random stream.
Points must be bit-identical (NaN equal to NaN); offsets, gt_boxes (in their dtype) and gt_names must be equal."""
import pickle

import numpy as np
import pytest
import torch

from tests import gt_sampling_oracle as GS
from tests import parity_utils as PU
from tests import world_aug_oracle as WA

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32 = np.float32
CLASSES = ["car", "truck", "construction_vehicle", "bus", "trailer", "barrier", "motorcycle", "bicycle", "pedestrian",
           "traffic_cone"]
GROUPS = ["car:2", "truck:3", "construction_vehicle:7", "bus:4", "trailer:6", "barrier:2", "motorcycle:6", "bicycle:6",
          "pedestrian:2", "traffic_cone:2"]
WORLD = [PU.Cfg(NAME="random_world_flip", ALONG_AXIS_LIST=["x", "y"]),
         PU.Cfg(NAME="random_world_rotation", WORLD_ROT_ANGLE=[-0.78539816, 0.78539816]),
         PU.Cfg(NAME="random_world_scaling", WORLD_SCALE_RANGE=[0.95, 1.05])]


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(((a.view(np.int32) == b.view(np.int32)) | (np.isnan(a) & np.isnan(b))).all())


def _cfg(info, **kw):
    cfg = dict(NAME="gt_sampling", DB_INFO_PATH=[info], PREPARE={"filter_by_min_points": [f"{c}:5" for c in CLASSES],
                                                                  "filter_by_difficulty": [-1]},
               SAMPLE_GROUPS=GROUPS, NUM_POINT_FEATURES=5, REMOVE_EXTRA_WIDTH=[0.0, 0.0, 0.0], LIMIT_WHOLE_SCENE=True)
    cfg.update(kw)
    return PU.Cfg(cfg)


def _gt(rng, m, cols, dtype):
    boxes = np.concatenate([rng.uniform(-50, 50, (m, 2)), rng.uniform(-2, 0, (m, 1)), rng.uniform(0.5, 5, (m, 3)),
                            rng.uniform(-np.pi, np.pi, (m, 1)), rng.normal(0, 2, (m, cols - 7))], 1).astype(dtype)
    return boxes, np.array([CLASSES[i] for i in rng.integers(0, len(CLASSES), m)])


def _oracle(root, cfg, frames, boxes, names, masks, seed, world):
    """The reference's forward, frame by frame: gt_sampling, then the world steps with draws taken right after, then
    the heading limit_period of the tail."""
    ref = GS.DataBaseSampler(root, cfg, CLASSES)
    np.random.seed(seed)
    out = []
    for f, g, nm, m in zip(frames, boxes, names, masks):
        dd = ref({"points": f.copy(), "gt_boxes": g.copy(), "gt_names": nm.copy(), "gt_boxes_mask": m.copy()})
        p, gb = dd["points"], dd["gt_boxes"]
        if world:
            p, gb = WA.world_augment(p, gb, world, WA.draw_world_augmentations(world))
        else:
            gb = gb.copy()
            gb[:, 6] = WA.limit_period(gb[:, 6], offset=0.5, period=2 * np.pi)
        out.append((p, gb, dd["gt_names"], dd["_accepted"]))
    return out


def _device(root, cfg, frames, boxes, names, masks, seed, world, x_col):
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    aug = DataAugmentor([cfg] + world, class_names=CLASSES, root_path=root, x_col=x_col)
    raw = np.concatenate(frames)
    pts = np.concatenate([np.concatenate([np.full((f.shape[0], 1), b, F32), f], 1) for b, f in enumerate(frames)]) if x_col else raw
    offs = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)
    np.random.seed(seed)
    dd = {"points": _t(pts), "point_frame_offsets": _t(offs), "gt_boxes": [g.copy() for g in boxes],
          "gt_names": [n.copy() for n in names], "gt_boxes_mask": [m.copy() for m in masks]}
    return aug, aug.forward(dict(dd)), dd


def _compare(got, want, x_col):
    pts, offs = got["points"].cpu().numpy(), got["point_frame_offsets"].cpu().numpy()
    assert "gt_boxes_mask" not in got and offs[0] == 0 and offs[-1] == pts.shape[0]
    for b, (p, gb, nm, _) in enumerate(want):
        rows = pts[offs[b]:offs[b + 1]]
        if x_col:
            assert np.all(rows[:, 0] == b)
        assert _bits_equal(rows[:, x_col:], p), f"frame {b}: points differ"
        assert got["gt_boxes"][b].dtype == gb.dtype and np.array_equal(got["gt_boxes"][b], gb), f"frame {b}: gt_boxes differ"
        assert list(np.asarray(got["gt_names"][b]).astype(str)) == list(np.asarray(nm).astype(str)), f"frame {b}: gt_names"


@pytest.fixture(scope="module")
def db_root(tmp_path_factory):
    roots = {}
    for dtype in (np.float32, np.float64):
        root = str(tmp_path_factory.mktemp("gtdb"))
        roots[np.dtype(dtype).name] = (root, GS.write_database(root, CLASSES, 60, 5, seed=11, box_dtype=dtype))
    return roots


@pytest.mark.parametrize("world", [False, True])
@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("x_col", [0, 1])
def test_full_frames_match_the_reference(db_root, x_col, dtype, world):
    from toda_b200 import synth
    root, info = db_root[dtype]
    cfg = _cfg(info)
    rng = np.random.default_rng(7)
    frames = [synth.make_frame("nus_0075", i) for i in range(4)]
    gt = [_gt(rng, m, 9, np.dtype(dtype)) for m in (25, 40, 8, 60)]
    boxes, names = [g[0] for g in gt], [g[1] for g in gt]
    masks = [rng.random(b.shape[0]) > 0.2 for b in boxes]
    steps = WORLD if world else []
    want = _oracle(root, cfg, frames, boxes, names, masks, 31, steps)
    aug, got, inputs = _device(root, cfg, frames, boxes, names, masks, 31, steps, x_col)
    _compare(got, want, x_col)
    assert sum(int(w[3].sum()) for w in want) > 20 and sum(int((~w[3]).sum()) for w in want) > 0
    # replaying the recorded draws gives the same result; a second run with the same seed is bit-identical
    again = aug.forward(dict(inputs, world_aug_draws=got["world_aug_draws"]))
    assert torch.equal(again["points"], got["points"]) and torch.equal(again["point_frame_offsets"], got["point_frame_offsets"])
    assert all(np.array_equal(a, b) for a, b in zip(again["gt_boxes"], got["gt_boxes"]))
    _, twice, _ = _device(root, cfg, frames, boxes, names, masks, 31, steps, x_col)
    assert torch.equal(twice["points"], got["points"])


def test_edge_cases(db_root, tmp_path):
    """A frame without gt boxes, an empty frame, a frame whose samples all collide with a gt box, and a database whose
    samples collide only with each other (every object of a class at one place)."""
    from toda_b200 import synth
    root, info = db_root["float32"]
    cfg = _cfg(info, LIMIT_WHOLE_SCENE=False)
    rng = np.random.default_rng(8)
    full = synth.make_frame("nus_0075", 5)
    frames = [full[:50000], full[:0], full[50000:90000], full[90000:]]
    cover = np.array([[0, 0, 0, 500, 500, 20, 0, 0, 0]], F32)
    b0, n0 = _gt(rng, 12, 9, F32)
    boxes = [np.zeros((0, 9), F32), b0, cover, np.zeros((0, 9), F32)]
    names = [np.array([], "<U20"), n0, np.array(["car"]), np.array([], "<U20")]
    masks = [np.zeros(b.shape[0], bool) | True for b in boxes]
    for x_col in (0, 1):
        want = _oracle(root, cfg, frames, boxes, names, masks, 5, [])
        assert not want[2][3].any()                                          # every sample collides with the cover box
        _, got, _ = _device(root, cfg, frames, boxes, names, masks, 5, [], x_col)
        _compare(got, want, x_col)
    # samples that collide only with each other: all cars of the database at one spot, two drawn per frame
    info2 = GS.write_database(str(tmp_path), CLASSES, 20, 5, seed=12)
    with open(tmp_path / info2, "rb") as f:
        infos = pickle.load(f)
    for i in infos["car"]:
        i["box3d_lidar"][:3] = [20.0, -20.0, -1.0]
    with open(tmp_path / info2, "wb") as f:
        pickle.dump(infos, f)
    cfg2 = _cfg(info2, LIMIT_WHOLE_SCENE=False, PREPARE={}, SAMPLE_GROUPS=["car:2", "pedestrian:3"])
    want = _oracle(str(tmp_path), cfg2, frames, boxes, names, masks, 6, [])
    assert all(not w[3][:2].any() for w, b in zip(want, boxes) if b is not cover)
    _, got, _ = _device(str(tmp_path), cfg2, frames, boxes, names, masks, 6, [], 1)
    _compare(got, want, 1)


def test_accepted_flags_on_near_contact_pairs():
    """12 000 sample / gt pairs that touch within a few centimetres (edge to edge, corner to corner, the 1e-2 margin
    and just outside it): the accepted flags equal the restatement's (iou row max == 0)."""
    from toda_b200 import ops
    rng = np.random.default_rng(21)
    batch, k = 24, 500
    gts, samples = [], []
    for b in range(batch):
        g = np.zeros((k, 7), F32)
        s = np.zeros((k, 7), F32)
        grid = np.stack(np.meshgrid(np.arange(40), np.arange(25)), -1).reshape(-1, 2)[:k] * 60.0 - 600.0
        g[:, :2] = grid
        g[:, 2] = rng.uniform(-1, 1, k)
        g[:, 3:6] = rng.uniform(0.3, 8, (k, 3))
        g[:, 6] = rng.uniform(-np.pi, np.pi, k)
        s[:, 2:6] = np.c_[rng.uniform(-1, 1, k), rng.uniform(0.3, 8, (k, 3))]
        mode = rng.integers(0, 3, k)
        gap = rng.choice([0.0, 1e-6, -1e-6, 0.005, -0.005, 0.0099, 0.0101, 0.02, -0.02], k) + rng.normal(0, 1e-3, k) * (mode == 2)
        # mode 0: side by side along the gt box's x axis, same heading (+- a hair); 1: along y, heading + pi/2;
        # 2: a random heading, the sample's centre at the gt box's corner distance
        hx, hy = g[:, 3] / 2, g[:, 4] / 2
        c, sn = np.cos(g[:, 6]), np.sin(g[:, 6])
        s[:, 6] = np.where(mode == 0, g[:, 6] + rng.choice([0, 1e-7, -1e-7], k), np.where(mode == 1, g[:, 6] + np.pi / 2,
                                                                                        rng.uniform(-np.pi, np.pi, k)))
        along = np.where(mode == 0, hx + s[:, 3] / 2 + gap, np.where(mode == 1, 0, hx + gap))
        side = np.where(mode == 1, hy + s[:, 3] / 2 + gap, np.where(mode == 2, hy + gap, 0))
        s[:, 0] = g[:, 0] + along * c - side * sn
        s[:, 1] = g[:, 1] + along * sn + side * c
        gts.append(g)
        samples.append(s)
    sampled = np.concatenate(samples)
    pts = _t(np.zeros((batch * 10, 5), F32))
    offs = _t(np.arange(0, batch * 10 + 1, 10, dtype=np.int32))
    rows = np.zeros((sampled.shape[0], 2), np.int64)
    _, _, acc = ops.gt_sampling(pts, offs, gts, sampled, np.full((batch, 1), k), _t(np.zeros((1, 5), F32)), rows,
                                np.zeros((sampled.shape[0], 3)), False, [0, 0, 0], x_col=0)
    want = np.concatenate([(GS.boxes_bev_iou_cpu(s, np.concatenate([g, s])) * (1 - np.eye(k, 2 * k, k, dtype=F32))).max(1) == 0
                           for g, s in zip(gts, samples)])
    assert 0.1 < want.mean() < 0.9, want.mean()
    assert np.array_equal(acc, want), int((acc != want).sum())


def test_sample_cap_is_reported():
    from toda_b200 import ops
    pts, offs = _t(np.zeros((4, 5), F32)), _t(np.array([0, 4], np.int32))
    n = ops.GTS_MAX_SAMPLES_PER_FRAME + 1
    with pytest.raises(RuntimeError, match="sampled boxes"):
        ops.gt_sampling(pts, offs, [np.zeros((0, 7), F32)], np.zeros((n, 7), F32), [[n]], _t(np.zeros((1, 5), F32)),
                        np.zeros((n, 2), np.int64), np.zeros((n, 3)), False, [0, 0, 0])


def test_pipeline_preprocess_equals_inline(db_root):
    """InputPipeline(preprocess=DataAugmentor with gt_sampling) gives the points, offsets and voxels of the same
    augmentation run in-line."""
    from tests.test_gpu_pipeline import _batches, _modules
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    from toda_b200.pipeline import InputPipeline
    dev = torch.device("cuda", 0)
    root, info = db_root["float32"]
    vfe, net, hc, pcr = _modules(dev, "fp32")
    aug = DataAugmentor([_cfg(info)] + WORLD, class_names=CLASSES, root_path=root)
    host = _batches(pcr, 3)
    rng = np.random.default_rng(2)
    gt = [[_gt(rng, 10, 9, F32) for _ in range(2)] for _ in host]

    def bd(i, p, o):
        return {"points": p, "point_frame_offsets": o, "batch_size": 2, "gt_boxes": [g[0].copy() for g in gt[i]],
                "gt_names": [g[1].copy() for g in gt[i]]}
    np.random.seed(9)
    want = [vfe(aug.forward(bd(i, p.to(dev), o.to(dev)))) for i, (p, o) in enumerate(host)]
    draws = [w["world_aug_draws"] for w in want]
    pipe = InputPipeline(vfe, net, dev, reserve_bytes=64 << 20, preprocess=aug.forward)
    for i, (p, o) in enumerate(host):
        got = pipe.consume(pipe.submit(dict(bd(i, p.pin_memory(), o.pin_memory()), world_aug_draws=draws[i])))
        for key in ("points", "point_frame_offsets", "voxels", "voxel_coords", "voxel_num_points"):
            assert torch.equal(got[key], want[i][key]), key
        assert all(np.array_equal(a, b) for a, b in zip(got["gt_boxes"], want[i]["gt_boxes"]))
    torch.cuda.synchronize()
