"""tests/rotate_paste_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU restatement of PolarMix's public rotate_copy and instance paste (Xiao et al., "PolarMix: A General Data
Augmentation Technique for LiDAR Point Clouds", NeurIPS 2022), as TODA's inter_domain_point_polarmix.py L153-191 uses it
for rotate-pasting, adapted to boxes with the collision rule this code base already pins for gt_sampling
(tests/gt_sampling_oracle.py: boxes_bev_iou_cpu of iou3d_cpu.cpp, points_in_boxes_cpu of roiaware_pool3d.cpp).  TODA's
file was not available when this was written: this restatement is the pin, and tests/test_oracle_rotate_paste.py checks
it against hand-derived cases.  If TODA's file later shows a difference, this module is what gets corrected.

For one frame, with the destination points and boxes, the source points, the source instance boxes (already filtered by
class) and a list of angles drawn by the caller ([0, w1, w2] reproduces PolarMix's `pts_copy = [pts_inst] + rotated
copies`):
  1. candidates: for each angle in list order and each instance box in order, the box rotated about z:
     x', y' = float32((x*R[0][j] + y*R[1][j]) + z*R[2][j]) evaluated in float64 without FMA, with PolarMix's float64
     rot_mat R = [[cos w, sin w, 0], [-sin w, cos w, 0], [0, 0, 1]] (np.cos / np.sin of the scalar angle); z unchanged;
     heading + w in float32, no period wrap; the velocity columns 7, 8 by the same 2x2 expression; other columns copied;
  2. collision, angle by angle: a candidate is accepted iff its iou_bev is exactly 0 against every destination box,
     every candidate accepted under an earlier angle and every other candidate of its own angle (gt_sampling's
     iou1.max + iou2.max == 0, iou1 = iou2 when there is no box yet), so two copies of one angle that collide are both
     dropped;
  3. instance points of box j: the source rows inside the unrotated, unenlarged box (check_pt_in_box3d_cpu), in source
     order; a row inside two instance boxes belongs to both;
  4. paste: the destination rows, all of them, in input order (PolarMix removes nothing), then for every accepted
     candidate in candidate order its instance rows with xyz rotated by the expression of step 1 rounded to float32 and
     every other column copied bit for bit.  PolarMix's public segmentation code, as recalled (not checked against a
     copy), copies only the intensity column of the rotated points and zeroes the rest; that is deliberately not
     reproduced here;
  5. boxes and names: the destination ones, then those of the accepted candidates.
PolarMix rotates with np.dot(xyz, rot_mat), whose float64 products BLAS may fuse; the elementwise form is pinned instead
because it does not depend on the BLAS build.  After rounding to float32 the two agree except where the elementwise
float64 value is exactly halfway between two float32 values, which takes a sum that cancelled down to 24 significant
bits: there the fused value can round one ulp the other way (1 coordinate in 3.3 million on the synthetic frames;
tests/test_oracle_rotate_paste.py checks that every disagreement is such a tie).
Only tests/ and scripts/ import this.
"""
import numpy as np

from tests import gt_sampling_oracle as GS

F32, F64 = np.float32, np.float64


def rot_mat(w):
    """PolarMix's rotation matrix of the angle w (float64)."""
    return np.array([[np.cos(w), np.sin(w), 0], [-np.sin(w), np.cos(w), 0], [0, 0, 1]])


def rotate_xyz(xyz, w):
    """float32 (N, 3) rotated about z: float32((x*R[0][j] + y*R[1][j]) + z*R[2][j]) in float64, op by op."""
    R = rot_mat(w)
    d = np.asarray(xyz, F32).astype(F64)
    out = np.empty(d.shape, F32)
    for j in range(3):
        out[:, j] = ((d[:, 0] * R[0, j] + d[:, 1] * R[1, j]) + d[:, 2] * R[2, j]).astype(F32)
    return out


def rotate_boxes(boxes, w):
    """Step 1: the candidate boxes of one angle, float32 (M, C)."""
    R = rot_mat(w)
    out = np.array(boxes, dtype=F32, copy=True).reshape(-1, np.shape(boxes)[-1])
    d = out[:, :3].astype(F64)
    for j in range(2):
        out[:, j] = ((d[:, 0] * R[0, j] + d[:, 1] * R[1, j]) + d[:, 2] * R[2, j]).astype(F32)
    out[:, 6] = out[:, 6] + F32(w)
    if out.shape[1] >= 9:
        v = out[:, 7:9].astype(F64)
        for j in range(2):
            out[:, 7 + j] = (v[:, 0] * R[0, j] + v[:, 1] * R[1, j]).astype(F32)
    return out


def instance_masks(points, inst_boxes):
    """Step 3: for each instance box, the bool mask of the (N, 3+) float32 points inside it."""
    return [GS.points_in_boxes_count(points[:, :3], inst_boxes[j:j + 1, :7]) > 0 for j in range(inst_boxes.shape[0])]


def rotate_paste_frame(dst_points, src_points, dst_boxes, dst_names, inst_boxes, inst_names, angles):
    """One frame, raw (N, F) float32 points with x, y, z in columns 0..2.  Returns (points, boxes, names, accepted), with
    accepted the bool flags of the candidates in candidate order (angle by angle)."""
    inst = np.asarray(inst_boxes).reshape(-1, np.shape(inst_boxes)[-1])
    existed = np.asarray(dst_boxes, F32).reshape(-1, np.shape(dst_boxes)[-1])[:, :7]
    masks = instance_masks(np.asarray(src_points, F32), inst.astype(F32))
    pasted, cand_all, accepted = [], [], []
    for w in angles:
        cand = rotate_boxes(inst, w)
        cand_all.append(cand)
        if cand.shape[0] == 0:
            continue
        iou1 = GS.boxes_bev_iou_cpu(cand[:, :7], existed)
        iou2 = GS.boxes_bev_iou_cpu(cand[:, :7], cand[:, :7])
        iou2[range(cand.shape[0]), range(cand.shape[0])] = 0
        iou1 = iou1 if iou1.shape[1] > 0 else iou2
        ok = (iou1.max(axis=1) + iou2.max(axis=1)) == 0
        accepted.append(ok)
        existed = np.concatenate([existed, cand[ok, :7]], axis=0)
        for j in np.nonzero(ok)[0]:
            rows = np.array(src_points[masks[j]], F32, copy=True)
            rows[:, :3] = rotate_xyz(rows[:, :3], w)
            pasted.append(rows)
    ok = np.concatenate(accepted) if accepted else np.zeros(0, bool)
    cands = np.concatenate(cand_all) if cand_all else np.zeros((0, inst.shape[1]), F32)
    points = np.concatenate([np.asarray(dst_points, F32)] + pasted, axis=0)
    boxes = np.concatenate([np.asarray(dst_boxes), cands[ok]], axis=0)
    names = np.concatenate([np.asarray(dst_names), np.tile(np.asarray(inst_names), len(angles))[ok]])
    return points, boxes, names, ok
