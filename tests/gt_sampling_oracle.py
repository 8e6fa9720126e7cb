"""tests/gt_sampling_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU restatement of pcdet's gt_sampling, restated from OpenPCDet v0.5.2: DataBaseSampler (__init__, filter_by_difficulty,
filter_by_min_points, sample_with_fixed_number, __call__, add_sampled_boxes_to_scene;
pcdet/datasets/augmentor/database_sampler.py), box_utils.enlarge_box3d / remove_points_in_boxes3d, and the compiled ops
they call (iou3d_cpu.cpp boxes_iou_bev_cpu, roiaware_pool3d.cpp points_in_boxes_cpu), the latter restated in C in
tests/gt_sampling_box_ops.c and compiled on first use (gcc -O2 -ffp-contract=off, as oracle/build.py compiles the
voxelizer's restatement) into a temporary directory, so a read-only tree works.  The oracle of the gt_sampling kernels
and of toda_b200.pcdet_plugin's gt_sampling step.  No reference checkout was available: this restatement is the pin, and
tests/test_oracle_gt_sampling.py checks it against hand-derived cases.  The behaviour it keeps from the reference, quirks included:
  - existed_boxes starts as the frame's UNMASKED gt_boxes; classes run in SAMPLE_GROUPS order (classes not in
    class_names are skipped), each tested against existed_boxes, which grows by the accepted boxes of earlier classes
    (iou1), and against its own samples with the diagonal zeroed (iou2); iou1 = iou2 when no box exists; a sample is
    accepted iff iou1.max + iou2.max == 0, so two samples that collide with each other are both dropped;
  - LIMIT_WHOLE_SCENE sets sample_num = SAMPLE_CLASS_NUM - (count of the class in the original gt_names), kept (as a
    string) in the group state;
  - sample_with_fixed_number redraws np.random.permutation only when pointer >= len; a slice past the end returns fewer
    than sample_num entries;
  - sampled boxes are cast to float32; the IoU and the point test see float32 boxes and points; enlarge_box3d enlarges
    in float32 torch;
  - object points are shifted by info['box3d_lidar'][:3] with numpy's in-place += (float64 database boxes: computed in
    float64, rounded to float32);
  - if any sample is accepted, gt_boxes / gt_names become the MASKED originals followed by the accepted samples, and the
    points the object points (acceptance order) followed by the surviving scene points; in every case gt_boxes_mask is
    popped, so the augmentor's tail does not apply it again.
Only tests/ and scripts/ import this.
"""
import atexit
import copy
import ctypes
import os
import pickle
import shutil
import subprocess
import tempfile

import numpy as np
import torch

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "gt_sampling_box_ops.c")
_lib = None


def _box_lib():
    global _lib
    if _lib is None:
        tmp = tempfile.mkdtemp(prefix="gt_sampling_oracle_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libgt_sampling_box_ops.so")
        subprocess.check_call(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC", "-o", so, _SRC, "-lm"])
        _lib = ctypes.CDLL(so)
        _lib.boxes_iou_bev_cpu.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
        _lib.box_overlap.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        _lib.box_overlap.restype = ctypes.c_float
        _lib.points_in_boxes_cpu.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_long, ctypes.c_int,
                                             ctypes.c_void_p]
    return _lib


def _f32(a):
    """check_numpy_to_torch(...).float(): a contiguous float32 copy."""
    return np.ascontiguousarray(np.asarray(a), dtype=np.float32)


def box_overlap(box_a, box_b):
    """iou3d_cpu.cpp box_overlap of two float32 (7,) boxes."""
    a, b = _f32(box_a), _f32(box_b)
    return float(_box_lib().box_overlap(a.ctypes.data, b.ctypes.data))


def boxes_bev_iou_cpu(boxes_a, boxes_b):
    """iou3d_nms_utils.boxes_bev_iou_cpu: (Na, 7) x (Nb, 7) -> float32 (Na, Nb)."""
    a, b = _f32(boxes_a), _f32(boxes_b)
    out = np.zeros((a.shape[0], b.shape[0]), np.float32)
    _box_lib().boxes_iou_bev_cpu(a.ctypes.data, a.shape[0], b.ctypes.data, b.shape[0], out.ctypes.data)
    return out


def points_in_boxes_count(points, boxes):
    """roiaware_pool3d_utils.points_in_boxes_cpu(points[:, 0:3], boxes) summed over the boxes: per point, the number of
    float32 (7,) boxes that contain it."""
    p, b = _f32(points), _f32(boxes)
    out = np.zeros(p.shape[0], np.int32)
    _box_lib().points_in_boxes_cpu(b.ctypes.data, b.shape[0], p.ctypes.data, p.shape[0], p.shape[1], out.ctypes.data)
    return out


def enlarge_box3d(boxes3d, extra_width=(0, 0, 0)):
    """box_utils.enlarge_box3d: float32 torch, sizes += extra_width (returned as numpy here)."""
    boxes = torch.from_numpy(np.ascontiguousarray(boxes3d)).float()
    large = boxes.clone()
    large[:, 3:6] += boxes.new_tensor(extra_width)[None, :]
    return large.numpy()


def remove_points_in_boxes3d(points, boxes3d):
    """box_utils.remove_points_in_boxes3d: the (float32) points outside every box."""
    points = _f32(points)
    return points[points_in_boxes_count(points, boxes3d) == 0]


def _get(cfg, key, default=None):
    return cfg.get(key, default)


class DataBaseSampler:
    """database_sampler.DataBaseSampler for the configs without USE_ROAD_PLANE / DATABASE_WITH_FAKELIDAR."""

    def __init__(self, root_path, sampler_cfg, class_names):
        self.root_path = root_path
        self.class_names = class_names
        self.sampler_cfg = sampler_cfg
        self.db_infos = {c: [] for c in class_names}
        self.use_shared_memory = _get(sampler_cfg, "USE_SHARED_MEMORY", False)
        for db_info_path in sampler_cfg["DB_INFO_PATH"]:
            with open(os.path.join(root_path, db_info_path), "rb") as f:
                infos = pickle.load(f)
                [self.db_infos[cur_class].extend(infos[cur_class]) for cur_class in class_names]
        for func_name, val in sampler_cfg["PREPARE"].items():
            self.db_infos = getattr(self, func_name)(self.db_infos, val)
        self.gt_database_data = (np.load(os.path.join(root_path, sampler_cfg["DB_DATA_PATH"][0]))
                                 if self.use_shared_memory else None)
        self.sample_groups = {}
        self.sample_class_num = {}
        self.limit_whole_scene = _get(sampler_cfg, "LIMIT_WHOLE_SCENE", False)
        for x in sampler_cfg["SAMPLE_GROUPS"]:
            class_name, sample_num = x.split(":")
            if class_name not in class_names:
                continue
            self.sample_class_num[class_name] = sample_num
            self.sample_groups[class_name] = {"sample_num": sample_num, "pointer": len(self.db_infos[class_name]),
                                              "indices": np.arange(len(self.db_infos[class_name]))}

    def filter_by_difficulty(self, db_infos, removed_difficulty):
        return {key: [info for info in dinfos if info["difficulty"] not in removed_difficulty]
                for key, dinfos in db_infos.items()}

    def filter_by_min_points(self, db_infos, min_gt_points_list):
        for name_num in min_gt_points_list:
            name, min_num = name_num.split(":")
            min_num = int(min_num)
            if min_num > 0 and name in db_infos.keys():
                db_infos[name] = [info for info in db_infos[name] if info["num_points_in_gt"] >= min_num]
        return db_infos

    def sample_with_fixed_number(self, class_name, sample_group):
        sample_num, pointer, indices = int(sample_group["sample_num"]), sample_group["pointer"], sample_group["indices"]
        if pointer >= len(self.db_infos[class_name]):
            indices = np.random.permutation(len(self.db_infos[class_name]))
            pointer = 0
        sampled_dict = [self.db_infos[class_name][idx] for idx in indices[pointer: pointer + sample_num]]
        pointer += sample_num
        sample_group["pointer"] = pointer
        sample_group["indices"] = indices
        return sampled_dict

    def add_sampled_boxes_to_scene(self, data_dict, sampled_gt_boxes, total_valid_sampled_dict):
        gt_boxes_mask = data_dict["gt_boxes_mask"]
        gt_boxes = data_dict["gt_boxes"][gt_boxes_mask]
        gt_names = data_dict["gt_names"][gt_boxes_mask]
        points = data_dict["points"]
        obj_points_list = []
        for info in total_valid_sampled_dict:
            if self.use_shared_memory:
                start_offset, end_offset = info["global_data_offset"]
                obj_points = copy.deepcopy(self.gt_database_data[start_offset:end_offset])
            else:
                file_path = os.path.join(self.root_path, info["path"])
                obj_points = np.fromfile(str(file_path), dtype=np.float32).reshape([-1, self.sampler_cfg["NUM_POINT_FEATURES"]])
            obj_points[:, :3] += info["box3d_lidar"][:3]
            obj_points_list.append(obj_points)
        obj_points = np.concatenate(obj_points_list, axis=0)
        sampled_gt_names = np.array([x["name"] for x in total_valid_sampled_dict])
        large_sampled_gt_boxes = enlarge_box3d(sampled_gt_boxes[:, 0:7], extra_width=self.sampler_cfg["REMOVE_EXTRA_WIDTH"])
        points = remove_points_in_boxes3d(points, large_sampled_gt_boxes)
        points = np.concatenate([obj_points, points], axis=0)
        gt_names = np.concatenate([gt_names, sampled_gt_names], axis=0)
        gt_boxes = np.concatenate([gt_boxes, sampled_gt_boxes], axis=0)
        data_dict["gt_boxes"] = gt_boxes
        data_dict["gt_names"] = gt_names
        data_dict["points"] = points
        return data_dict

    def __call__(self, data_dict):
        """data_dict: points (N, F) float32, gt_boxes (M, 7+), gt_names (M,), gt_boxes_mask (M,) bool.  Also records the
        accepted flags of every sample (in sampling order) as data_dict['_accepted'] for the tests."""
        gt_boxes = data_dict["gt_boxes"]
        gt_names = data_dict["gt_names"].astype(str)
        existed_boxes = gt_boxes
        total_valid_sampled_dict = []
        accepted = []
        for class_name, sample_group in self.sample_groups.items():
            if self.limit_whole_scene:
                num_gt = np.sum(class_name == gt_names)
                sample_group["sample_num"] = str(int(self.sample_class_num[class_name]) - num_gt)
            if int(sample_group["sample_num"]) > 0:
                sampled_dict = self.sample_with_fixed_number(class_name, sample_group)
                sampled_boxes = np.stack([x["box3d_lidar"] for x in sampled_dict], axis=0).astype(np.float32)
                iou1 = boxes_bev_iou_cpu(sampled_boxes[:, 0:7], existed_boxes[:, 0:7])
                iou2 = boxes_bev_iou_cpu(sampled_boxes[:, 0:7], sampled_boxes[:, 0:7])
                iou2[range(sampled_boxes.shape[0]), range(sampled_boxes.shape[0])] = 0
                iou1 = iou1 if iou1.shape[1] > 0 else iou2
                ok = (iou1.max(axis=1) + iou2.max(axis=1)) == 0
                accepted.append(ok)
                valid_mask = ok.nonzero()[0]
                valid_sampled_dict = [sampled_dict[x] for x in valid_mask]
                valid_sampled_boxes = sampled_boxes[valid_mask]
                existed_boxes = np.concatenate((existed_boxes, valid_sampled_boxes), axis=0)
                total_valid_sampled_dict.extend(valid_sampled_dict)
        sampled_gt_boxes = existed_boxes[gt_boxes.shape[0]:, :]
        if total_valid_sampled_dict.__len__() > 0:
            data_dict = self.add_sampled_boxes_to_scene(data_dict, sampled_gt_boxes, total_valid_sampled_dict)
        data_dict.pop("gt_boxes_mask")
        data_dict["_accepted"] = np.concatenate(accepted) if accepted else np.zeros(0, bool)
        return data_dict


def write_database(root, class_names, per_class, num_features, seed, box_dtype=np.float32, velocity=True, shared=False):
    """A small database in pcdet's format under `root`: gt_database/<class>_<i>.bin files (or, with shared, one
    gt_database_global.npy with global_data_offset), and dbinfos.pkl.  Objects sit around the origin of their box (the
    database stores them relative to the box centre); sizes, points and difficulty vary.  Returns the info-pickle name."""
    rng = np.random.default_rng(seed)
    os.makedirs(os.path.join(root, "gt_database"), exist_ok=True)
    infos, stacked, row = {}, [], 0
    sizes = {"car": (4.5, 1.9, 1.6), "truck": (7.0, 2.5, 3.0), "construction_vehicle": (6.0, 2.8, 3.2), "bus": (11.0, 2.9, 3.5),
             "trailer": (12.0, 2.9, 3.8), "barrier": (0.5, 2.5, 1.0), "motorcycle": (2.1, 0.8, 1.5), "bicycle": (1.7, 0.6, 1.3),
             "pedestrian": (0.7, 0.7, 1.8), "traffic_cone": (0.4, 0.4, 1.0)}
    for c in class_names:
        infos[c] = []
        base = np.array(sizes.get(c, (2.0, 1.0, 1.5)))
        for i in range(per_class):
            size = base * rng.uniform(0.8, 1.2, 3)
            centre = np.array([rng.uniform(-50, 50), rng.uniform(-50, 50), rng.uniform(-2.0, 0.5)])
            box = np.concatenate([centre, size, [rng.uniform(-np.pi, np.pi)]] + ([rng.normal(0, 2, 2)] if velocity else []))
            m = int(rng.integers(0, 300)) if i % 7 else 0
            pts = np.concatenate([rng.uniform(-0.5, 0.5, (m, 3)) * size, rng.random((m, num_features - 3))], 1).astype(np.float32)
            path = os.path.join("gt_database", f"{c}_{i}.bin")
            info = {"name": c, "path": path, "box3d_lidar": box.astype(box_dtype), "num_points_in_gt": m,
                    "difficulty": int(rng.integers(0, 3)), "gt_idx": i, "image_idx": i}
            if shared:
                info["global_data_offset"] = [row, row + m]
                stacked.append(pts)
                row += m
            else:
                pts.tofile(os.path.join(root, path))
            infos[c].append(info)
    with open(os.path.join(root, "dbinfos.pkl"), "wb") as f:
        pickle.dump(infos, f)
    if shared:
        np.save(os.path.join(root, "gt_database_global.npy"), np.concatenate(stacked).astype(np.float32))
    return "dbinfos.pkl"
