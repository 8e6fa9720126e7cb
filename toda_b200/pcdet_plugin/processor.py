"""GPU counterpart of the point side of pcdet's DataProcessor and of TODA's point mixers.

Mirrors, for device-resident batches, the reference's host pre-steps that sit immediately before voxelization
(SURVEY.md section 8 rows a-0, a-0b, a-2 and f-1), so raw frames need to cross PCIe once:

    DataProcessor.mask_points_and_boxes_outside_range   pcdet/datasets/processor/data_processor.py L78-91  (points part)
    DataProcessor.shuffle_points                        data_processor.py L93-103
    DatasetTemplate.collate_batch, 'points' key         pcdet/datasets/dataset.py L173-178
    inter_domain_point_cutmix, points part              pcdet/datasets/processor/inter_domain_point_cutmix.py L45-69
    swap (PolarMix), points part                        inter_domain_point_polarmix.py L72-95
    intra_domain_point_mixup, points part               intra_domain_point_mixup.py L23-27

Random decisions stay where the reference makes them (numpy on the host: permutations, lambda, crop rectangle, sector
angles) and are passed in, which is what makes the results comparable row for row; `shuffle_points` falls back to a
device permutation when none is given.  gt_boxes handling (a few hundred boxes) stays on the host.
"""
from functools import partial

import numpy as np
import torch

from .. import ops


class PointPreprocessor:
    """Same two-phase protocol as the reference (`getattr(self, cfg.NAME)(config=cfg)` at init, then per batch) over a
    device batch: data_dict['points'] (sum N, 1+F) = [b, x, y, z, ...] and data_dict['point_frame_offsets'] int32 (B+1)."""

    def __init__(self, processor_configs, point_cloud_range, training, num_point_features):
        self.point_cloud_range = np.asarray(point_cloud_range, dtype=np.float32)
        self.training = training
        self.num_point_features = num_point_features
        self.mode = "train" if training else "test"
        self.grid_size = self.voxel_size = None
        self.data_processor_queue = []
        for step_cfg in processor_configs:
            name = step_cfg["NAME"] if isinstance(step_cfg, dict) else step_cfg.NAME
            step = getattr(self, name, None)
            if step is None:
                raise NotImplementedError(f"PointPreprocessor has no step {name!r} (voxelization happens in the VFE: use "
                                          "transform_points_to_voxels_placeholder)")
            self.data_processor_queue.append(step(config=step_cfg))      # phase 1: bind the config, get the per-batch callable

    @staticmethod
    def _get(cfg, key, default=None):
        return cfg.get(key, default) if hasattr(cfg, "get") else getattr(cfg, key, default)

    def mask_points_and_boxes_outside_range(self, data_dict=None, config=None):
        if data_dict is None:
            return partial(self.mask_points_and_boxes_outside_range, config=config)
        if data_dict.get("points", None) is not None:
            r = self.point_cloud_range
            pts, offs = ops.points_select(data_dict["points"], data_dict.get("point_frame_offsets"), ops.SELECT_RANGE_XY,
                                          [r[0], r[1], r[3], r[4]], x_col=1)
            data_dict["points"] = pts
            if data_dict.get("point_frame_offsets") is not None:
                data_dict["point_frame_offsets"] = offs
        return data_dict

    def shuffle_points(self, data_dict=None, config=None):
        if data_dict is None:
            return partial(self.shuffle_points, config=config)
        enabled = self._get(config, "SHUFFLE_ENABLED")
        if enabled[self.mode]:
            points = data_dict["points"]
            idx = data_dict.pop("shuffle_idx", None)       # per-batch row permutation that keeps frames contiguous
            if idx is None:
                idx = self._device_permutation(points, data_dict.get("point_frame_offsets"))
            elif not torch.is_tensor(idx):
                idx = torch.as_tensor(np.asarray(idx), dtype=torch.int32, device=points.device)
            data_dict["points"] = ops.gather_point_rows(points, idx.int().contiguous())
        return data_dict

    @staticmethod
    def _device_permutation(points, offsets):
        n = points.shape[0]
        if offsets is None:
            return torch.randperm(n, device=points.device).int()
        # shuffle inside every frame: sort random keys that carry the frame index in their integer part
        key = torch.rand(n, device=points.device, dtype=torch.float64) + points[:, 0].double()
        return torch.argsort(key).int()

    def transform_points_to_voxels_placeholder(self, data_dict=None, config=None):
        """Voxelization itself happens in the VFE (K1); this step only publishes grid_size / voxel_size, as the
        reference's placeholder does (data_processor.py L105-113)."""
        if data_dict is not None:
            return data_dict
        self.voxel_size = self._get(config, "VOXEL_SIZE")
        self.grid_size = ops.grid_size_xyz(self.point_cloud_range, self.voxel_size)
        return partial(self.transform_points_to_voxels_placeholder, config=config)

    def forward(self, data_dict):
        for step in self.data_processor_queue:                            # phase 2: run the bound steps in cfg order
            data_dict = step(data_dict=data_dict)
        return data_dict


def collate_points(raw_points, frame_offsets):
    """collate_batch's 'points' branch on the device: raw frames (sum N, F) stored back to back + int32 offsets (B+1) ->
    (sum N, 1+F) with the frame index in column 0.  (A range mask that keeps everything: one fused pass.)"""
    inf = float("inf")
    out, _ = ops.points_select(raw_points, frame_offsets, ops.SELECT_RANGE_XY, [-inf, -inf, inf, inf], add_batch_col=True,
                               x_col=0, trim=False)
    return out


def cutmix_points(source_points, target_points, min_xy, max_xy, x_col=0):
    """Target points strictly inside the crop rectangle, then source points outside it."""
    rect = [float(min_xy[0]), float(min_xy[1]), float(max_xy[0]), float(max_xy[1])]
    inside_t, _ = ops.points_select(target_points, None, ops.SELECT_RECT_XY, rect, x_col=x_col)
    outside_s, _ = ops.points_select(source_points, None, ops.SELECT_RECT_XY, rect, invert=True, x_col=x_col)
    return torch.cat([inside_t, outside_s], dim=0)


def polar_swap_points(pt1, pt2, start_angle, end_angle, dis_th=None, dis_less=True, x_col=0):
    """pt1 without its [start, end] sector, then pt2's sector (swap(); with dis_th: swap_with_range's point masks)."""
    dm = 0 if dis_th is None else (1 if dis_less else 2)
    p = [float(start_angle), float(end_angle), float(dis_th or 0.0), float(dm)]
    keep1, _ = ops.points_select(pt1, None, ops.SELECT_SECTOR, p, invert=True, x_col=x_col)
    take2, _ = ops.points_select(pt2, None, ops.SELECT_SECTOR, p, x_col=x_col)
    return torch.cat([keep1, take2], dim=0)


def rotation_cos_sin(angles):
    """(A, 2) float64 (cos w, sin w) of each angle, as PolarMix's rot_mat takes them (np.cos / np.sin of the scalar)."""
    return np.array([[np.cos(w), np.sin(w)] for w in np.asarray(angles, np.float64).reshape(-1)], np.float64).reshape(-1, 2)


def rotate_boxes_about_z(boxes, cos_sin, angle):
    """Boxes (M, 7 / 9 / 10) rotated about z: x, y as float32((x*R[0][j] + y*R[1][j]) + z*R[2][j]) in float64 without FMA
    with R = [[c, s, 0], [-s, c, 0], [0, 0, 1]], z unchanged, heading + angle in float32 (no period wrap), the velocity
    columns 7, 8 by the same 2x2 expression, any other column copied.  Returns float32 (M, C)."""
    src = np.asarray(boxes)
    out = src.astype(np.float32, copy=True)
    c, s = float(cos_sin[0]), float(cos_sin[1])
    r = np.array([[c, s, 0.0], [-s, c, 0.0], [0.0, 0.0, 1.0]])
    x, y, z = (out[:, k].astype(np.float64) for k in range(3))
    for k in range(2):
        out[:, k] = ((x * r[0, k] + y * r[1, k]) + z * r[2, k]).astype(np.float32)
    out[:, 6] = out[:, 6] + np.float32(angle)
    if out.shape[1] >= 9:
        vx, vy = out[:, 7].astype(np.float64), out[:, 8].astype(np.float64)
        out[:, 7] = (vx * r[0, 0] + vy * r[1, 0]).astype(np.float32)
        out[:, 8] = (vx * r[0, 1] + vy * r[1, 1]).astype(np.float32)
    return out


def rotate_paste_points(dst_points, dst_offsets, src_points, src_offsets, gt_boxes, gt_names, inst_boxes, inst_names, angles,
                        x_col=0):
    """PolarMix's rotate-pasting (rotate_copy + paste, inter_domain_point_polarmix.py L153-191) for a batch of frames,
    adapted to boxes: frame b's instance boxes inst_boxes[b] (M_b, 7 / 9 / 10 columns, already filtered by class) are
    copied, rotated about z by each angle of angles[b] (drawn by the caller; [0, w1, w2] reproduces PolarMix's
    `[pts_inst] + rotated copies`), the copies whose BEV IoU with a box already in the scene is not exactly 0 are dropped
    (gt_sampling's rule, angle by angle, see include/toda_b200.h), and the source points inside the instance box of each
    surviving copy are appended to the destination frame, rotated by its angle.

    dst_points / src_points (N, x_col + F) float32 CUDA with frame offsets int32 (B+1) CUDA (src may be dst).  gt_boxes,
    gt_names: the destination frames' boxes and names (per-frame host arrays); inst_names: the names of the instance boxes.
    Returns (points, frame_offsets, boxes, names): boxes[b] / names[b] are the destination boxes / names followed by those
    of the accepted copies, in angle order and, within an angle, instance order.
    """
    batch = len(gt_boxes)
    inst = [np.asarray(m).reshape(-1, np.shape(m)[-1]) for m in inst_boxes]
    for b, m in enumerate(inst):
        if m.shape[1] not in (7, 9, 10) or np.shape(gt_boxes[b])[-1] != m.shape[1]:
            raise ValueError(f"rotate_paste_points: frame {b} has instance boxes of {m.shape[1]} columns and destination "
                             f"boxes of {np.shape(gt_boxes[b])[-1]} (7, 9 or 10, the same on both sides)")
    if not len(gt_names) == len(inst) == len(inst_names) == len(angles) == batch:
        raise ValueError(f"rotate_paste_points: {batch} frames need {batch} name arrays, instance tables and angle lists")
    rotations = [rotation_cos_sin(a) for a in angles]
    cands = [np.concatenate([rotate_boxes_about_z(m, cs, w) for cs, w in zip(r, np.asarray(a, np.float64).reshape(-1))])
             if len(r) else np.zeros((0, m.shape[1]), np.float32) for m, r, a in zip(inst, rotations, angles)]
    points, offsets, accepted = ops.rotate_paste(dst_points, dst_offsets, src_points, src_offsets, gt_boxes, inst, cands,
                                                 rotations, x_col=x_col)
    boxes, names, lo = [], [], 0
    for b in range(batch):
        ok = accepted[lo:lo + cands[b].shape[0]]
        lo += cands[b].shape[0]
        boxes.append(np.concatenate([np.asarray(gt_boxes[b]), cands[b][ok]], axis=0))
        names.append(np.concatenate([np.asarray(gt_names[b]), np.tile(np.asarray(inst_names[b]), len(rotations[b]))[ok]]))
    return points, offsets, boxes, names


def mixup_points(points_1, points_2, lam, shuffle_idx_1, shuffle_idx_2):
    """Prefixes int(N1*lam) / int(N2*(1-lam)) of the two shuffled frames."""
    def prefix(points, idx, frac):
        k = int(points.shape[0] * frac)
        idx = torch.as_tensor(np.asarray(idx[:k]), dtype=torch.int32, device=points.device) if not torch.is_tensor(idx) else idx[:k].int()
        return ops.gather_point_rows(points, idx.contiguous())
    return torch.cat([prefix(points_1, shuffle_idx_1, lam), prefix(points_2, shuffle_idx_2, 1 - lam)], dim=0)


def _box_params(boxes, margin):
    """params of TODA_SELECT_BOXES: [M, margin, M x (cx, cy, cz, dx, dy, dz, rz)] from (M, >= 7) boxes (extra columns, e.g. the
    class index of gt_boxes, are dropped); values are float32, as the reference's gt_boxes are."""
    b = torch.as_tensor(boxes, dtype=torch.float32).cpu()
    b = b.reshape(-1, b.shape[-1])[:, :7]
    return [float(b.shape[0]), float(margin)] + [float(v) for v in b.reshape(-1).tolist()]


def points_in_boxes(points, boxes, margin=1e-1, x_col=0):
    """Rows of `points` that lie in ANY of `boxes` (N_box <= 96, (cx, cy, cz, dx, dy, dz, rz[, ...]) rows), input order kept:
    the union of augmentor_utils.get_points_in_box (pcdet/datasets/augmentor/augmentor_utils.py L474-491) over the boxes.
    The boxes (a few dozen floats) are read on the host, as the reference reads them."""
    n_box = int(boxes.shape[0])
    if n_box > ops.SELECT_MAX_BOXES:
        raise ValueError("points_in_boxes: at most %d boxes per call" % ops.SELECT_MAX_BOXES)
    out, _ = ops.points_select(points, None, ops.SELECT_BOXES, _box_params(boxes, margin), x_col=x_col)
    return out


def remove_points_in_boxes(points, boxes, margin=1e-1, x_col=0):
    """The point filter of intra_domain_point_mixup_cd (intra_domain_point_mixup.py L50-59): drop every point that lies in
    any of `boxes`.  More than 96 boxes are applied in chunks (removal composes)."""
    n_box = int(boxes.shape[0])
    for lo in range(0, max(n_box, 1), ops.SELECT_MAX_BOXES):
        chunk = boxes[lo:lo + ops.SELECT_MAX_BOXES]
        if chunk.shape[0] == 0:
            break
        points, _ = ops.points_select(points, None, ops.SELECT_BOXES, _box_params(chunk, margin), invert=True, x_col=x_col)
    return points
