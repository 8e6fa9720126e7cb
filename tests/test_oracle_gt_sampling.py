"""The gt_sampling restatement (tests/gt_sampling_oracle.py, tests/gt_sampling_box_ops.c; OpenPCDet v0.5.2) against hand-derived
cases, the plugin's sampler state and database loader against the restatement, and the config protocol -- runs on CPU."""
import os

import numpy as np
import pytest

from tests import gt_sampling_oracle as GS
from tests import parity_utils as PU

F32 = np.float32
NUS_CLASSES = ["car", "truck", "construction_vehicle", "bus", "trailer", "barrier", "motorcycle", "bicycle", "pedestrian",
               "traffic_cone"]


def _box(x, y, dx, dy, h=0.0, z=0.0, dz=2.0):
    return np.array([x, y, z, dx, dy, dz, h], F32)


def test_box_overlap_hand_derived():
    a = _box(0, 0, 2, 2)
    assert GS.box_overlap(a, _box(5, 0, 2, 2)) == 0                                    # disjoint
    assert GS.box_overlap(_box(0, 0, 4, 4), a) == 4 and GS.box_overlap(a, _box(0, 0, 4, 4)) == 4   # containment
    assert GS.box_overlap(_box(1, 2, 2, 3), _box(1, 2, 2, 3)) == 6                      # identical boxes
    octagon = 8 * (np.sqrt(2) - 1)                                                      # two unit squares at 45 degrees
    assert abs(GS.box_overlap(a, _box(0, 0, 2, 2, np.pi / 4)) - octagon) < 1e-5
    assert abs(GS.box_overlap(_box(0, 0, 2, 2, np.pi / 4), a) - octagon) < 1e-5
    assert GS.box_overlap(a, _box(2, 0, 2, 2)) == 0                                     # edge contact: a line, no area
    assert GS.box_overlap(a, _box(2.005, 2.005, 2, 2)) == 0                             # corners inside the 1e-2 margin only
    assert abs(GS.box_overlap(a, _box(1.995, 1.995, 2, 2)) - 0.005 ** 2) < 1e-6        # a real 5 mm x 5 mm overlap
    assert GS.box_overlap(a, _box(1.5, 0, 1, 1, np.pi / 2)) == 0                        # rotated, edge contact at x = 1
    assert abs(GS.box_overlap(a, _box(1.25, 0, 2, 1, np.pi / 2)) - 0.5) < 1e-5          # rotated, 0.25 x 2 overlap
    # rotated edge contact: cos(pi/2) is not 0 in float32, the corners land off the line and a rounding-sized area
    # remains, so the reference rejects such a sample
    assert 0 < GS.box_overlap(a, _box(1.5, 0, 2, 1, np.pi / 2)) < 1e-6


def test_iou_and_point_test():
    boxes = np.stack([_box(0, 0, 2, 2), _box(1, 0, 2, 2), _box(10, 0, 2, 2)])
    iou = GS.boxes_bev_iou_cpu(boxes, boxes)
    assert iou.dtype == F32 and np.allclose(np.diag(iou), 1) and abs(iou[0, 1] - 2 / 6) < 1e-6 and iou[0, 2] == 0
    pts = np.array([[0, 0, 0], [0.995, 0, 0], [1.0099, 0, 0], [1.0101, 0, 0], [0, 0, 1.0], [0, 0, 1.01]], F32)
    # |local| < d / 2 + 1e-2 in x, y; |z - cz| <= dz / 2 (no margin)
    assert GS.points_in_boxes_count(pts, boxes[:1]).tolist() == [1, 1, 1, 0, 1, 0]
    big = GS.enlarge_box3d(boxes[:1], [0.5, 0.5, 0.5])
    assert big.dtype == F32 and big[0, 3:6].tolist() == [2.5, 2.5, 2.5]
    assert GS.remove_points_in_boxes3d(pts, big).shape[0] == 0


def _cfg(root, info, groups, **kw):
    cfg = dict(NAME="gt_sampling", DB_INFO_PATH=[info], PREPARE={}, SAMPLE_GROUPS=groups, NUM_POINT_FEATURES=5,
               REMOVE_EXTRA_WIDTH=[0.0, 0.0, 0.0], LIMIT_WHOLE_SCENE=False)
    cfg.update(kw)
    return PU.Cfg(cfg)


def test_sampler_state_machine(tmp_path):
    """sample_with_fixed_number: a permutation at the first draw and whenever pointer >= len; a slice that runs past the
    end is short.  The plugin's draws equal the restatement's, group by group, with LIMIT_WHOLE_SCENE counting the
    frame's original gt_names."""
    from toda_b200.pcdet_plugin.augmentor import _GtSampling
    info = GS.write_database(str(tmp_path), ["car", "bus"], 5, 5, seed=1)
    for limit in (False, True):
        cfg = _cfg(str(tmp_path), info, ["car:3", "bus:2", "bicycle:4"], LIMIT_WHOLE_SCENE=limit)
        ref = GS.DataBaseSampler(str(tmp_path), cfg, ["car", "bus"])
        step = _GtSampling(cfg, ["car", "bus"], str(tmp_path))
        assert [g[0] for g in step.groups] == ["car", "bus"]
        frames = [np.array(["car"]), np.array([], str), np.array(["bus", "bus", "car"]), np.array(["car"] * 4)]
        np.random.seed(4)
        got = [step.draw(nm) for nm in frames * 2]
        np.random.seed(4)
        want = []
        for nm in frames * 2:
            d = []
            for c, g in ref.sample_groups.items():
                if limit:
                    g["sample_num"] = str(int(ref.sample_class_num[c]) - np.sum(c == nm.astype(str)))
                n0 = g["pointer"]
                d.append(np.array([ref.db_infos[c].index(x) for x in ref.sample_with_fixed_number(c, g)])
                         if int(g["sample_num"]) > 0 else np.zeros(0, int))
                if int(g["sample_num"]) > 0 and n0 < 5:
                    assert g["pointer"] == n0 + int(g["sample_num"])
            want.append(d)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert [x.tolist() for x in g] == [x.tolist() for x in w]
        if not limit:
            # car: 3 from a permutation, then the 2 left (short slice), then a new permutation
            assert [len(d[0]) for d in got[:3]] == [3, 2, 3]
            assert sorted(got[0][0].tolist() + got[1][0].tolist()) == list(range(5))
        else:
            assert [len(d[0]) for d in got[:4]] == [2, 3, 2, 0]                # 3 - count of car in the frame


def test_prepare_filters_and_loader(tmp_path):
    """PREPARE (filter_by_min_points, filter_by_difficulty) as the reference applies them; the loader reads the same
    objects and points from the .bin files and from the shared .npy."""
    from toda_b200.pcdet_plugin import database
    classes = ["car", "pedestrian", "bus"]
    for shared in (False, True):
        root = str(tmp_path / ("shm" if shared else "bin"))
        info = GS.write_database(root, classes, 12, 5, seed=2, shared=shared, box_dtype=np.float64)
        prep = {"filter_by_min_points": ["car:50", "pedestrian:1", "bus:0"], "filter_by_difficulty": [1]}
        cfg = _cfg(root, info, ["car:2"], PREPARE=prep, USE_SHARED_MEMORY=shared, DB_DATA_PATH=["gt_database_global.npy"])
        ref = GS.DataBaseSampler(root, cfg, classes[:2])
        host = database.parse_database(root, cfg, classes[:2])
        assert host.box_dtype == np.float64
        for c in classes[:2]:
            assert [i["gt_idx"] for i in host.infos[c]] == [i["gt_idx"] for i in ref.db_infos[c]]
            assert all(i["difficulty"] != 1 for i in host.infos[c])
            assert np.array_equal(host.boxes[c], np.stack([i["box3d_lidar"] for i in ref.db_infos[c]]))
            for k, i in enumerate(ref.db_infos[c]):
                if shared:
                    want = ref.gt_database_data[i["global_data_offset"][0]:i["global_data_offset"][1]]
                else:
                    want = np.fromfile(os.path.join(root, i["path"]), F32).reshape(-1, 5)
                r0, n = host.first_row[c][k], host.num_rows[c][k]
                assert np.array_equal(host.points[r0:r0 + n], want)
        assert all(i["num_points_in_gt"] >= 50 for i in host.infos["car"])
        assert all(i["num_points_in_gt"] >= 1 for i in host.infos["pedestrian"])
        assert "bus" not in host.infos
        with pytest.raises(NotImplementedError, match="USE_ROAD_PLANE"):
            database.parse_database(root, _cfg(root, info, ["car:2"], USE_ROAD_PLANE=True), classes)
        with pytest.raises(NotImplementedError, match="DATABASE_WITH_FAKELIDAR"):
            database.parse_database(root, _cfg(root, info, ["car:2"], DATABASE_WITH_FAKELIDAR=True), classes)


def test_oracle_mask_quirk_and_acceptance(tmp_path):
    """A frame whose samples all collide keeps its UNMASKED gt_boxes and loses gt_boxes_mask; a frame with accepted
    samples gets the masked gt_boxes followed by the samples, and the object points in front of the kept points."""
    info = GS.write_database(str(tmp_path), ["car"], 3, 5, seed=3, velocity=False)
    cfg = _cfg(str(tmp_path), info, ["car:3"])
    ref = GS.DataBaseSampler(str(tmp_path), cfg, ["car"])
    pts = (np.random.default_rng(0).random((500, 5)) * 100 - 50).astype(F32)
    cover = np.array([[0, 0, 0, 200, 200, 10, 0]], F32)                                # every sample collides with it
    np.random.seed(0)
    dd = ref({"points": pts, "gt_boxes": cover.copy(), "gt_names": np.array(["car"]), "gt_boxes_mask": np.array([False])})
    assert "gt_boxes_mask" not in dd and dd["gt_boxes"].shape[0] == 1 and not dd["_accepted"].any()
    assert dd["points"] is pts
    far = np.array([[500, 500, 0, 1, 1, 1, 0], [600, 600, 0, 1, 1, 1, 0]], F32)
    dd = ref({"points": pts, "gt_boxes": far.copy(), "gt_names": np.array(["car", "car"]), "gt_boxes_mask": np.array([False, True])})
    acc = dd["_accepted"]
    assert acc.sum() >= 1 and dd["gt_boxes"].shape[0] == 1 + acc.sum() and np.array_equal(dd["gt_boxes"][0], far[1])
    assert list(dd["gt_names"]) == ["car"] * (1 + acc.sum())


def test_augmentor_config_protocol_with_gt_sampling(tmp_path):
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    info = GS.write_database(str(tmp_path), NUS_CLASSES, 4, 5, seed=5)
    gts = _cfg(str(tmp_path), info, [f"{c}:2" for c in NUS_CLASSES])
    flip = PU.Cfg(NAME="random_world_flip", ALONG_AXIS_LIST=["x"])
    with pytest.raises(NotImplementedError, match="gt_sampling"):
        DataAugmentor([gts, flip], class_names=NUS_CLASSES)                           # no root_path
    with pytest.raises(NotImplementedError, match="gt_sampling"):
        DataAugmentor([gts, flip], root_path=str(tmp_path))                           # no class_names
    aug = DataAugmentor(PU.Cfg(AUG_CONFIG_LIST=[gts, flip], DISABLE_AUG_LIST=[]), class_names=NUS_CLASSES[:3],
                        root_path=str(tmp_path))
    assert [s.name for s in aug.data_augmentor_queue] == ["gt_sampling", "random_world_flip"]
    assert [g[0] for g in aug.data_augmentor_queue[0].groups] == NUS_CLASSES[:3]
    assert len(DataAugmentor([gts, flip], host_steps=["gt_sampling"]).data_augmentor_queue) == 1
    with pytest.raises(NotImplementedError, match="USE_ROAD_PLANE"):
        DataAugmentor([PU.Cfg(dict(gts, USE_ROAD_PLANE=True))], class_names=NUS_CLASSES, root_path=str(tmp_path))
