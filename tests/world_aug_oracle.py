"""tests/world_aug_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU restatement of the world augmentations of pcdet's DataAugmentor, restated from OpenPCDet v0.5.2
(pcdet/datasets/augmentor/data_augmentor.py L43-80, augmentor_utils.py L8-82, common_utils.rotate_points_along_z /
limit_period): the oracle for K0's world transform (`toda_points_world_transform`) and for
toda_b200.pcdet_plugin.augmentor.DataAugmentor.  Each augmentor_utils function takes its random draw as an argument;
draw_world_augmentations makes the draws in the reference's order.  No reference checkout was available to generate
goldens from the reference's own functions: this restatement is the pin, and tests/test_oracle_augment.py checks it
against hand-derived cases and against torch's CPU matmul dispatch.  Only tests/ and scripts/ import this.
"""
import numpy as np
import torch


def rotate_points_along_z(points, angle):
    """common_utils.rotate_points_along_z for (B, N, 3+C) points and (B,) angles: everything converted to float32 torch
    (check_numpy_to_torch calls .float()), cos / sin in float32, xyz @ [[c, s, 0], [-s, c, 0], [0, 0, 1]] with torch.matmul
    on the CPU, the other columns appended unchanged."""
    pts = torch.from_numpy(np.ascontiguousarray(points)).float()
    ang = torch.from_numpy(np.asarray(angle)).float()
    cosa, sina = torch.cos(ang), torch.sin(ang)
    zeros, ones = ang.new_zeros(pts.shape[0]), ang.new_ones(pts.shape[0])
    rot = torch.stack((cosa, sina, zeros, -sina, cosa, zeros, zeros, zeros, ones), dim=1).view(-1, 3, 3).float()
    out = torch.matmul(pts[:, :, 0:3], rot)
    return torch.cat((out, pts[:, :, 3:]), dim=-1).numpy()


def limit_period(val, offset=0.5, period=np.pi):
    """common_utils.limit_period on a numpy array (float32 torch)."""
    v = torch.from_numpy(np.ascontiguousarray(val)).float()
    return (v - torch.floor(v / period + offset) * period).numpy()


def random_flip_along_x(gt_boxes, points, enable):
    """augmentor_utils.random_flip_along_x with its draw `enable` given."""
    if enable:
        gt_boxes[:, 1] = -gt_boxes[:, 1]
        gt_boxes[:, 6] = -gt_boxes[:, 6]
        points[:, 1] = -points[:, 1]
        if gt_boxes.shape[1] > 7:
            gt_boxes[:, 8] = -gt_boxes[:, 8]
    return gt_boxes, points


def random_flip_along_y(gt_boxes, points, enable):
    """augmentor_utils.random_flip_along_y with its draw `enable` given."""
    if enable:
        gt_boxes[:, 0] = -gt_boxes[:, 0]
        gt_boxes[:, 6] = -(gt_boxes[:, 6] + np.pi)
        points[:, 0] = -points[:, 0]
        if gt_boxes.shape[1] > 7:
            gt_boxes[:, 7] = -gt_boxes[:, 7]
    return gt_boxes, points


def global_rotation(gt_boxes, points, noise_rotation):
    """augmentor_utils.global_rotation with its draw `noise_rotation` given."""
    points = rotate_points_along_z(points[np.newaxis, :, :], np.array([noise_rotation]))[0]
    gt_boxes[:, 0:3] = rotate_points_along_z(gt_boxes[np.newaxis, :, 0:3], np.array([noise_rotation]))[0]
    gt_boxes[:, 6] += noise_rotation
    if gt_boxes.shape[1] > 7:
        gt_boxes[:, 7:9] = rotate_points_along_z(
            np.hstack((gt_boxes[:, 7:9], np.zeros((gt_boxes.shape[0], 1))))[np.newaxis, :, :],
            np.array([noise_rotation]))[0][:, 0:2]
    return gt_boxes, points


def global_scaling(gt_boxes, points, noise_scale):
    """augmentor_utils.global_scaling with its draw given (None when the range is narrower than 1e-3: nothing happens)."""
    if noise_scale is None:
        return gt_boxes, points
    points[:, :3] *= noise_scale
    gt_boxes[:, :6] *= noise_scale
    return gt_boxes, points


def draw_world_augmentations(step_configs):
    """The draws one frame consumes, in the reference's order: per step of the config list, random_world_flip draws
    np.random.choice([False, True], replace=False, p=[0.5, 0.5]) per axis of ALONG_AXIS_LIST, random_world_rotation
    np.random.uniform over WORLD_ROT_ANGLE (a scalar r means [-r, r]), random_world_scaling np.random.uniform over
    WORLD_SCALE_RANGE unless the range is narrower than 1e-3 (no draw, None)."""
    draws = []
    for cfg in step_configs:
        if cfg["NAME"] == "random_world_flip":
            draws.append([np.random.choice([False, True], replace=False, p=[0.5, 0.5]) for _ in cfg["ALONG_AXIS_LIST"]])
        elif cfg["NAME"] == "random_world_rotation":
            rot_range = cfg["WORLD_ROT_ANGLE"]
            if not isinstance(rot_range, list):
                rot_range = [-rot_range, rot_range]
            draws.append(np.random.uniform(rot_range[0], rot_range[1]))
        else:
            scale_range = cfg["WORLD_SCALE_RANGE"]
            draws.append(None if scale_range[1] - scale_range[0] < 1e-3 else np.random.uniform(scale_range[0], scale_range[1]))
    return draws


def world_augment(points, gt_boxes, step_configs, draws):
    """DataAugmentor.forward over the world steps for one frame with recorded draws: the steps in config order, then the
    heading limit_period of the forward's tail.  Returns new (points, gt_boxes)."""
    points, gt_boxes = np.array(points, copy=True), np.array(gt_boxes, copy=True)
    for cfg, d in zip(step_configs, draws):
        if cfg["NAME"] == "random_world_flip":
            for axis, enable in zip(cfg["ALONG_AXIS_LIST"], d):
                flip = random_flip_along_x if axis == "x" else random_flip_along_y
                gt_boxes, points = flip(gt_boxes, points, enable)
        elif cfg["NAME"] == "random_world_rotation":
            gt_boxes, points = global_rotation(gt_boxes, points, d)
        else:
            gt_boxes, points = global_scaling(gt_boxes, points, d)
    gt_boxes[:, 6] = limit_period(gt_boxes[:, 6], offset=0.5, period=2 * np.pi)
    return points, gt_boxes
