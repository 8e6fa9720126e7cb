"""GPU counterpart of the world augmentations of pcdet's DataAugmentor (OpenPCDet v0.5.2):

    DataAugmentor.random_world_flip / random_world_rotation / random_world_scaling
        pcdet/datasets/augmentor/data_augmentor.py L43-80
    augmentor_utils.random_flip_along_x / _y, global_rotation, global_scaling
        pcdet/datasets/augmentor/augmentor_utils.py L8-82
    DataAugmentor.forward, tail (heading limit_period, gt_boxes_mask)

    DataBaseSampler (gt_sampling)
        pcdet/datasets/augmentor/database_sampler.py (__init__, sample_with_fixed_number, __call__,
        add_sampled_boxes_to_scene)

The reference runs these per frame on the DataLoader workers.  Here the points of a whole batch are transformed on the
device by one launch of K0's world transform, bit-identical to the reference's float32 arithmetic, and gt_sampling's
collision test, scene-point removal and paste run on the device from a device-resident database (database.py).  As for
the mixers (processor.py), the random draws are made on the host with np.random in the reference's order, and gt_boxes
(a few dozen rows per frame) are transformed on the host with the reference's own expressions.
"""
import numpy as np
import torch

from .. import ops
from . import database

_WORLD_STEPS = ("random_world_flip", "random_world_rotation", "random_world_scaling")


def _get(cfg, key, default=None):
    return cfg.get(key, default) if hasattr(cfg, "get") else getattr(cfg, key, default)


def _rotate_points_along_z(points, angle):
    """common_utils.rotate_points_along_z for one (N, 3+C) array and one angle: float32 torch on the CPU, as there."""
    pts = torch.from_numpy(np.ascontiguousarray(points)[np.newaxis]).float()
    angle = torch.from_numpy(np.array([angle])).float()
    cosa, sina = torch.cos(angle), torch.sin(angle)
    zeros, ones = angle.new_zeros(1), angle.new_ones(1)
    rot = torch.stack((cosa, sina, zeros, -sina, cosa, zeros, zeros, zeros, ones), dim=1).view(-1, 3, 3).float()
    out = torch.matmul(pts[:, :, 0:3], rot)
    return torch.cat((out, pts[:, :, 3:]), dim=-1)[0].numpy()


def _limit_period(val, offset=0.5, period=np.pi):
    """common_utils.limit_period on a numpy array (converted to float32 torch, as check_numpy_to_torch does)."""
    v = torch.from_numpy(np.ascontiguousarray(val)).float()
    return (v - torch.floor(v / period + offset) * period).numpy()


class _Step:
    """One bound world step: `draw()` makes the frame's random draws in the reference's order, `point_ops` turns the
    draws of every frame into kernel steps, `boxes` applies one frame's draw to its gt_boxes."""

    def __init__(self, name, config):
        self.name, self.config = name, config
        if name == "random_world_flip":
            self.axes = list(_get(config, "ALONG_AXIS_LIST"))
            for a in self.axes:
                if a not in ("x", "y"):
                    raise ValueError(f"random_world_flip: axis {a!r} is not 'x' or 'y'")
        elif name == "random_world_rotation":
            r = _get(config, "WORLD_ROT_ANGLE")
            self.range = list(r) if isinstance(r, (list, tuple)) else [-r, r]
        else:
            self.range = list(_get(config, "WORLD_SCALE_RANGE"))
            self.active = self.range[1] - self.range[0] >= 1e-3       # global_scaling returns before drawing otherwise

    def draw(self):
        if self.name == "random_world_flip":
            return [bool(np.random.choice([False, True], replace=False, p=[0.5, 0.5])) for _ in self.axes]
        if self.name == "random_world_scaling" and not self.active:
            return None
        return float(np.random.uniform(self.range[0], self.range[1]))

    def point_ops(self, draws):
        if self.name == "random_world_flip":
            return [(ops.WORLD_FLIP_X if a == "x" else ops.WORLD_FLIP_Y, [d[j] for d in draws]) for j, a in enumerate(self.axes)]
        if self.name == "random_world_rotation":
            # one angle per call, as rotate_points_along_z takes it: torch's vectorised cos / sin may round differently
            cs = []
            for d in draws:
                a = torch.from_numpy(np.array([d])).float()
                cs.append([torch.cos(a).item(), torch.sin(a).item()])
            return [(ops.WORLD_ROTATE, cs)]
        return [(ops.WORLD_SCALE, draws)] if self.active else []

    def boxes(self, gt_boxes, d):
        if self.name == "random_world_flip":
            for axis, enable in zip(self.axes, d):
                if not enable:
                    continue
                if axis == "x":                                             # random_flip_along_x
                    gt_boxes[:, 1] = -gt_boxes[:, 1]
                    gt_boxes[:, 6] = -gt_boxes[:, 6]
                    if gt_boxes.shape[1] > 7:
                        gt_boxes[:, 8] = -gt_boxes[:, 8]
                else:                                                       # random_flip_along_y
                    gt_boxes[:, 0] = -gt_boxes[:, 0]
                    gt_boxes[:, 6] = -(gt_boxes[:, 6] + np.pi)
                    if gt_boxes.shape[1] > 7:
                        gt_boxes[:, 7] = -gt_boxes[:, 7]
        elif self.name == "random_world_rotation":                          # global_rotation
            gt_boxes[:, 0:3] = _rotate_points_along_z(gt_boxes[:, 0:3], d)
            gt_boxes[:, 6] += d
            if gt_boxes.shape[1] > 7:
                vel = np.hstack((gt_boxes[:, 7:9], np.zeros((gt_boxes.shape[0], 1))))
                gt_boxes[:, 7:9] = _rotate_points_along_z(vel, d)[:, 0:2]
        elif d is not None:                                                 # global_scaling
            gt_boxes[:, :6] *= d
        return gt_boxes


class _GtSampling:
    """gt_sampling (DataBaseSampler) as a device step.  The sampler state (the per-class permutation and pointer) lives
    here, as in the reference's sampler object; `draw()` consumes np.random as sample_with_fixed_number does and returns
    the sampled database indices of every group (an empty array for a group that draws nothing)."""

    name = "gt_sampling"

    def __init__(self, config, class_names, root_path):
        self.config = config
        self.db = database.load_database(root_path, config, class_names)
        host = self.db["host"]
        self.limit_whole_scene = bool(_get(config, "LIMIT_WHOLE_SCENE", False))
        self.extra_width = np.asarray(_get(config, "REMOVE_EXTRA_WIDTH", (0.0, 0.0, 0.0)), np.float32)
        self.groups = []           # [class name, sample_num (a string, as the reference keeps it), pointer, indices]
        self.sample_class_num = {}
        for x in _get(config, "SAMPLE_GROUPS"):
            class_name, sample_num = x.split(":")
            if class_name not in class_names:
                continue
            self.sample_class_num[class_name] = sample_num
            n = len(host.infos[class_name])
            self.groups.append([class_name, sample_num, n, np.arange(n)])
        if len(self.groups) > ops.GTS_MAX_GROUPS:
            raise ValueError(f"gt_sampling: {len(self.groups)} sample groups (at most {ops.GTS_MAX_GROUPS})")

    def draw(self, gt_names):
        out = []
        names = np.asarray(gt_names).astype(str)
        for g in self.groups:
            class_name = g[0]
            if self.limit_whole_scene:
                g[1] = str(int(self.sample_class_num[class_name]) - np.sum(class_name == names))
            sample_num = int(g[1])
            if sample_num <= 0:
                out.append(np.zeros(0, np.int64))
                continue
            n = len(self.db["host"].infos[class_name])
            pointer, indices = g[2], g[3]
            if pointer >= n:                                          # sample_with_fixed_number
                indices = np.random.permutation(n)
                pointer = 0
            picked = np.asarray(indices[pointer:pointer + sample_num], np.int64)
            if picked.size == 0:
                raise ValueError(f"gt_sampling: the database has no {class_name!r} objects to sample")
            g[2], g[3] = pointer + sample_num, indices
            out.append(picked)
        return out

    def apply(self, points, offsets, x_col, boxes, names, mask, draws):
        """Runs the step for a batch with the frames' draws; returns (points, offsets, boxes, names)."""
        host = self.db["host"]
        if points.shape[1] - x_col != host.num_point_features:
            raise ValueError(f"gt_sampling: NUM_POINT_FEATURES is {host.num_point_features}, the frames have "
                             f"{points.shape[1] - x_col} features")
        sizes = np.array([[len(i) for i in d] for d in draws], np.int32)
        if sizes.sum() == 0:
            return points, offsets, boxes, names
        cls = [g[0] for g in self.groups]
        sel = [(c, i) for d in draws for c, i in zip(cls, d)]
        stored = np.concatenate([host.boxes[c][i] for c, i in sel])
        sampled = stored.astype(np.float32)
        rows = np.stack([np.concatenate([host.first_row[c][i] for c, i in sel]),
                         np.concatenate([host.num_rows[c][i] for c, i in sel])], 1)
        snames = np.concatenate([host.names[c][i] for c, i in sel])
        points, offsets, accepted = ops.gt_sampling(
            points, offsets, boxes, sampled, sizes, database.device_points(self.db, points.device), rows,
            stored[:, :3].astype(np.float64), host.box_dtype == np.float64, self.extra_width, x_col=x_col)
        first = np.cumsum([0] + sizes.sum(1).tolist())
        boxes, names = list(boxes), list(names)
        for b in range(len(draws)):
            acc = np.nonzero(accepted[first[b]:first[b + 1]])[0] + first[b]
            if acc.size == 0:
                continue
            m = slice(None) if mask is None else mask[b]
            boxes[b] = np.concatenate([boxes[b][m], sampled[acc]], axis=0)
            names[b] = np.concatenate([np.asarray(names[b])[m], snames[acc]], axis=0)
        return points, offsets, boxes, names


class DataAugmentor:
    """pcdet's DataAugmentor protocol (`getattr(self, cfg.NAME)(config=cfg)` at init, then `forward(data_dict)`) over a
    device batch, for the world steps.

    augmentor_configs: a list of step configs, or a config with AUG_CONFIG_LIST and DISABLE_AUG_LIST.  host_steps: names
    of steps the caller has already run on the host; they are skipped.  gt_sampling is a device step when root_path (the
    dataset root that DB_INFO_PATH / DB_DATA_PATH are relative to) and class_names are given; its database is read and
    uploaded once per process.  Any other step that is not a world step raises NotImplementedError.  x_col: column of x
    in data_dict['points'], 0 for raw frames (sum N, F), 1 for collated [b, x, y, z, ...].

    forward(data_dict) reads
      points               (sum N, stride) float32 CUDA, frames back to back
      point_frame_offsets  int32 (B+1) CUDA tensor (optional with one frame)
      gt_boxes             optional list of B host arrays (M_b, 7|9|10), float32 or float64 (required by gt_sampling)
      gt_names             list of B host arrays of class names (required by gt_sampling)
      gt_boxes_mask        optional list of B boolean arrays (applied to gt_boxes / gt_names, as the reference does;
                           gt_sampling applies it only to the frames that receive samples, and pops it)
      world_aug_draws      optional recorded draws, [frame][step], to replay instead of drawing
    and writes the transformed points (and point_frame_offsets when gt_sampling runs), the transformed gt_boxes (new
    arrays), gt_names and the draws it used.
    """

    def __init__(self, augmentor_configs, class_names=None, host_steps=(), x_col=1, root_path=None):
        self.class_names = class_names
        self.root_path = root_path
        self.x_col = x_col
        self.data_augmentor_queue = []
        is_list = isinstance(augmentor_configs, (list, tuple))
        cfg_list = augmentor_configs if is_list else _get(augmentor_configs, "AUG_CONFIG_LIST")
        disabled = [] if is_list else list(_get(augmentor_configs, "DISABLE_AUG_LIST", None) or [])
        for cur_cfg in cfg_list:
            name = _get(cur_cfg, "NAME")
            if name in disabled or name in host_steps:
                continue
            if name == "gt_sampling" and (root_path is None or class_names is None):
                raise NotImplementedError("DataAugmentor runs gt_sampling on the device only with root_path and class_names: "
                                          "pass them, or run it on the host and name it in host_steps")
            if name not in _WORLD_STEPS + ("gt_sampling",):
                raise NotImplementedError(f"DataAugmentor has no device step {name!r}: run it on the host and name it in "
                                          "host_steps, or list it in DISABLE_AUG_LIST")
            self.data_augmentor_queue.append(getattr(self, name)(config=cur_cfg))

    def gt_sampling(self, config=None):
        return _GtSampling(config, self.class_names, self.root_path)

    def random_world_flip(self, config=None):
        return _Step("random_world_flip", config)

    def random_world_rotation(self, config=None):
        return _Step("random_world_rotation", config)

    def random_world_scaling(self, config=None):
        return _Step("random_world_scaling", config)

    def forward(self, data_dict):
        points, offsets = data_dict["points"], data_dict.get("point_frame_offsets")
        batch = 1 if offsets is None else offsets.numel() - 1
        gt_boxes = data_dict.get("gt_boxes")
        if gt_boxes is not None and not isinstance(gt_boxes, (list, tuple)):
            raise ValueError("DataAugmentor: gt_boxes must be a list of per-frame (M_b, 7+) arrays; a collated, zero-padded "
                             "array would not keep its padding rows at zero")
        sampling = any(step.name == "gt_sampling" for step in self.data_augmentor_queue)
        names = data_dict.get("gt_names")
        if sampling and (gt_boxes is None or names is None or len(gt_boxes) != batch or len(names) != batch):
            raise ValueError(f"DataAugmentor: gt_sampling needs gt_boxes and gt_names, one array per frame ({batch} frames)")
        draws = data_dict.get("world_aug_draws")
        if draws is None:
            draws = [[step.draw(names[b]) if step.name == "gt_sampling" else step.draw() for step in self.data_augmentor_queue]
                     for b in range(batch)]                                                   # frame by frame
        if len(draws) != batch or any(len(d) != len(self.data_augmentor_queue) for d in draws):
            raise ValueError(f"DataAugmentor: world_aug_draws must hold {len(self.data_augmentor_queue)} draws for each of "
                             f"{batch} frames")
        if gt_boxes is not None:
            if len(gt_boxes) != batch:
                raise ValueError(f"DataAugmentor: {len(gt_boxes)} gt_boxes arrays for {batch} frames")
            gt_boxes = [np.array(boxes, copy=True) for boxes in gt_boxes]
        mask = data_dict.pop("gt_boxes_mask", None) if gt_boxes is not None else None
        if sampling and offsets is None:
            offsets = torch.tensor([0, points.shape[0]], dtype=torch.int32, device=points.device)
        # the point side: world steps in one transform launch per run of them, split around gt_sampling
        point_ops = []
        for s, step in enumerate(self.data_augmentor_queue):
            if step.name == "gt_sampling":
                if point_ops:
                    points = ops.points_world_transform(points, offsets, point_ops, x_col=self.x_col)
                    point_ops = []
                points, offsets, gt_boxes, names = step.apply(points, offsets, self.x_col, gt_boxes, names, mask,
                                                              [d[s] for d in draws])
                data_dict["point_frame_offsets"] = offsets
                continue
            point_ops += step.point_ops([d[s] for d in draws])
            if gt_boxes is not None:
                gt_boxes = [step.boxes(boxes, draws[b][s]) for b, boxes in enumerate(gt_boxes)]
        if point_ops or not sampling:
            points = ops.points_world_transform(points, offsets, point_ops, x_col=self.x_col)
        data_dict["points"] = points
        data_dict["world_aug_draws"] = draws
        if gt_boxes is not None:
            for boxes in gt_boxes:
                boxes[:, 6] = _limit_period(boxes[:, 6], offset=0.5, period=2 * np.pi)
            if mask is not None and not sampling:
                gt_boxes = [g[m] for g, m in zip(gt_boxes, mask)]
                if names is not None:
                    names = [np.asarray(nm)[m] for nm, m in zip(names, mask)]
            data_dict["gt_boxes"] = gt_boxes
            if names is not None:
                data_dict["gt_names"] = names
        return data_dict
