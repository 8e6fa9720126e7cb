"""GPU counterpart of the world augmentations of pcdet's DataAugmentor (OpenPCDet v0.5.2):

    DataAugmentor.random_world_flip / random_world_rotation / random_world_scaling
        pcdet/datasets/augmentor/data_augmentor.py L43-80
    augmentor_utils.random_flip_along_x / _y, global_rotation, global_scaling
        pcdet/datasets/augmentor/augmentor_utils.py L8-82
    DataAugmentor.forward, tail (heading limit_period, gt_boxes_mask)

The reference runs these per frame on the DataLoader workers.  Here the points of a whole batch are transformed on the
device by one launch of K0's world transform, bit-identical to the reference's float32 arithmetic.  As for the mixers
(processor.py), the random draws are made on the host with np.random in the reference's order, and gt_boxes (a few
dozen rows per frame) are transformed on the host with the reference's own expressions.
"""
import numpy as np
import torch

from .. import ops

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


class DataAugmentor:
    """pcdet's DataAugmentor protocol (`getattr(self, cfg.NAME)(config=cfg)` at init, then `forward(data_dict)`) over a
    device batch, for the world steps.

    augmentor_configs: a list of step configs, or a config with AUG_CONFIG_LIST and DISABLE_AUG_LIST.  host_steps: names
    of steps the caller has already run on the host (e.g. gt_sampling, which reads its database from disk); they are
    skipped.  Any other step that is not a world step raises NotImplementedError.  x_col: column of x in
    data_dict['points'], 0 for raw frames (sum N, F), 1 for collated [b, x, y, z, ...].

    forward(data_dict) reads
      points               (sum N, stride) float32 CUDA, frames back to back
      point_frame_offsets  int32 (B+1) CUDA tensor (optional with one frame)
      gt_boxes             optional list of B host arrays (M_b, 7|9|10), float32 or float64
      gt_boxes_mask        optional list of B boolean arrays (applied to gt_boxes / gt_names, as the reference does)
      world_aug_draws      optional recorded draws, [frame][step], to replay instead of drawing
    and writes the transformed points, the transformed gt_boxes (new arrays) and the draws it used.
    """

    def __init__(self, augmentor_configs, class_names=None, host_steps=(), x_col=1):
        self.class_names = class_names
        self.x_col = x_col
        self.data_augmentor_queue = []
        is_list = isinstance(augmentor_configs, (list, tuple))
        cfg_list = augmentor_configs if is_list else _get(augmentor_configs, "AUG_CONFIG_LIST")
        disabled = [] if is_list else list(_get(augmentor_configs, "DISABLE_AUG_LIST", None) or [])
        for cur_cfg in cfg_list:
            name = _get(cur_cfg, "NAME")
            if name in disabled or name in host_steps:
                continue
            if name not in _WORLD_STEPS:
                raise NotImplementedError(f"DataAugmentor has no device step {name!r}: run it on the host and name it in "
                                          "host_steps, or list it in DISABLE_AUG_LIST")
            self.data_augmentor_queue.append(getattr(self, name)(config=cur_cfg))

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
        draws = data_dict.get("world_aug_draws")
        if draws is None:
            draws = [[step.draw() for step in self.data_augmentor_queue] for _ in range(batch)]   # frame by frame
        if len(draws) != batch or any(len(d) != len(self.data_augmentor_queue) for d in draws):
            raise ValueError(f"DataAugmentor: world_aug_draws must hold {len(self.data_augmentor_queue)} draws for each of "
                             f"{batch} frames")
        point_ops = []
        for s, step in enumerate(self.data_augmentor_queue):
            point_ops += step.point_ops([d[s] for d in draws])
        data_dict["points"] = ops.points_world_transform(points, offsets, point_ops, x_col=self.x_col)
        data_dict["world_aug_draws"] = draws
        if gt_boxes is not None:
            if len(gt_boxes) != batch:
                raise ValueError(f"DataAugmentor: {len(gt_boxes)} gt_boxes arrays for {batch} frames")
            out = []
            for b, boxes in enumerate(gt_boxes):
                boxes = np.array(boxes, copy=True)
                for s, step in enumerate(self.data_augmentor_queue):
                    boxes = step.boxes(boxes, draws[b][s])
                boxes[:, 6] = _limit_period(boxes[:, 6], offset=0.5, period=2 * np.pi)
                out.append(boxes)
            mask = data_dict.pop("gt_boxes_mask", None)
            if mask is not None:
                out = [g[m] for g, m in zip(out, mask)]
                if data_dict.get("gt_names") is not None:
                    data_dict["gt_names"] = [np.asarray(nm)[m] for nm, m in zip(data_dict["gt_names"], mask)]
            data_dict["gt_boxes"] = out
        return data_dict
