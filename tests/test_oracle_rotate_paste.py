"""The rotate-paste restatement (tests/rotate_paste_oracle.py) against hand-derived cases, its elementwise rotation
against np.dot on the synthetic frames, and the plugin's host-side candidate boxes against the restatement -- runs on CPU."""
import numpy as np
import pytest

from tests import rotate_paste_oracle as RP

F32 = np.float32
EMPTY = np.zeros((0, 7), F32)
NONE = np.array([], "<U10")


def _box(x, y, dx=4.0, dy=2.0, h=0.0, z=0.0, dz=2.0):
    return np.array([x, y, z, dx, dy, dz, h], F32)


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool((a.view(np.int32) == b.view(np.int32)).all())


def _run(dst, src, dst_boxes, inst, angles, dst_names=None, inst_names=None):
    dst_names = NONE[:0] if dst_names is None else np.asarray(dst_names)
    inst_names = np.array(["car"] * len(inst)) if inst_names is None else np.asarray(inst_names)
    return RP.rotate_paste_frame(np.asarray(dst, F32).reshape(-1, 4), np.asarray(src, F32).reshape(-1, 4),
                                 np.asarray(dst_boxes, F32).reshape(-1, 7), dst_names, np.asarray(inst, F32).reshape(-1, 7),
                                 inst_names, angles)


def test_quarter_turn_moves_box_and_points():
    """A box at (10, 0) rotated by pi/2 lands at (0, 10) with heading +pi/2, and its points move with it."""
    src = np.array([[10, 0, 0.5, 1], [10.5, 0.25, -0.5, 2], [20, 0, 0, 3]], F32)
    pts, boxes, names, ok = _run(np.zeros((0, 4)), src, EMPTY, [_box(10, 0, h=0.1)], [np.pi / 2])
    assert ok.tolist() == [True] and names.tolist() == ["car"]
    assert abs(boxes[0, 0]) < 1e-6 and boxes[0, 1] == 10 and boxes[0, 2] == 0
    assert boxes[0, 6] == F32(0.1) + F32(np.pi / 2) and boxes[0, 3:6].tolist() == [4, 2, 2]
    assert pts.shape == (2, 4) and pts[:, 3].tolist() == [1, 2]          # the third row is outside the box
    assert np.allclose(pts[:, :3], [[0, 10, 0.5], [-0.25, 10.5, -0.5]], atol=1e-6)
    assert _bits_equal(pts[:, :3], np.dot(src[:2, :3], RP.rot_mat(np.pi / 2)).astype(F32))


def test_copy_on_a_destination_box_is_rejected():
    dst = np.array([[1, 1, 1, 1]], F32)
    src = np.array([[10, 0, 0, 7]], F32)
    pts, boxes, names, ok = _run(dst, src, [_box(0, 10, h=np.pi / 2)], [_box(10, 0)], [np.pi / 2, np.pi],
                                 dst_names=["truck"])
    assert ok.tolist() == [False, True]                                  # pi lands at (-10, 0), away from the truck
    assert names.tolist() == ["truck", "car"] and abs(boxes[1, 0] + 10) < 1e-5
    assert pts.shape == (2, 4) and _bits_equal(pts[0], dst[0]) and pts[1, 3] == 7


def test_overlapping_copies_of_one_angle_are_both_dropped():
    src = np.array([[10, 0, 0, 1], [11, 0, 0, 2]], F32)
    inst = [_box(10, 0), _box(11.5, 0), _box(-20, 0)]
    pts, boxes, names, ok = _run(np.zeros((0, 4)), src, EMPTY, inst, [0.3], inst_names=["a", "b", "c"])
    assert ok.tolist() == [False, False, True] and names.tolist() == ["c"] and pts.shape == (0, 4)


def test_copy_that_collides_only_with_an_earlier_angle_is_dropped():
    src = np.array([[10, 0, 0, 1]], F32)
    pts, boxes, names, ok = _run(np.zeros((0, 4)), src, EMPTY, [_box(10, 0)], [0.0, 0.01, np.pi])
    assert ok.tolist() == [True, False, True]
    assert pts.shape == (2, 4) and boxes.shape == (2, 7)


def test_zero_angle_is_an_unrotated_copy():
    """w = 0 with source != destination: PolarMix's unrotated instance copy, bit for bit."""
    dst = np.array([[-5, -5, -1, 9]], F32)
    src = np.array([[10.25, 0.5, 0.75, 1], [9.5, -0.3, -0.2, 2]], F32)
    inst = _box(10, 0, h=0.7)
    pts, boxes, _, ok = _run(dst, src, EMPTY, [inst], [0.0])
    assert ok.tolist() == [True] and _bits_equal(boxes[0], inst)
    assert _bits_equal(pts, np.concatenate([dst, src]))


def test_point_in_two_boxes_is_copied_twice_and_margin_points_are_copied():
    """Edge-to-edge boxes do not collide (area 0); the row on the shared edge is inside both (|local| < d/2 + 1e-2)."""
    src = np.array([[1.0, 0, 0, 1], [-1.005, 0, 0, 2], [3.009, 0, 0, 3], [3.02, 0, 0, 4], [0, 0, 1.01, 5]], F32)
    inst = [_box(0, 0, dx=2), _box(2, 0, dx=2)]
    pts, boxes, _, ok = _run(np.zeros((0, 4)), src, EMPTY, inst, [0.0])
    assert ok.tolist() == [True, True]
    assert pts[:, 3].tolist() == [1, 2, 1, 3]                            # z 1.01 > dz / 2 is outside: no z margin


def test_box_without_points_is_pasted_with_zero_rows():
    src = np.array([[10, 0, 0, 1]], F32)
    pts, boxes, names, ok = _run(np.zeros((0, 4)), src, EMPTY, [_box(30, 30), _box(10, 0)], [0.5], inst_names=["a", "b"])
    assert ok.tolist() == [True, True] and names.tolist() == ["a", "b"] and pts.shape == (1, 4)


def test_no_instances_or_no_angles_leave_the_frame_unchanged():
    dst = np.array([[1, 2, 3, 4]], F32)
    for inst, angles in ((np.zeros((0, 7), F32), [0.0, 1.0]), ([_box(10, 0)], [])):
        pts, boxes, names, ok = _run(dst, dst, [_box(-9, -9)], inst, angles, dst_names=["car"])
        assert ok.shape == (0,) and _bits_equal(pts, dst) and boxes.shape == (1, 7) and names.tolist() == ["car"]


def test_velocity_columns_rotate_and_other_columns_are_copied():
    b = np.array([[10, 0, -1, 4, 2, 1.5, 0.2, 3.0, 0.0, 7.0]], F32)
    c = RP.rotate_boxes(b, np.pi / 2)
    assert abs(c[0, 7]) < 1e-6 and c[0, 8] == 3 and c[0, 9] == 7 and c[0, 2] == -1 and _bits_equal(c[0, 3:6], b[0, 3:6])


def test_elementwise_rotation_agrees_with_np_dot_on_synthetic_frames():
    """PolarMix rotates with np.dot(xyz, rot_mat), whose float64 products BLAS may fuse.  After rounding to float32 the
    elementwise form agrees except where its float64 value is exactly halfway between two float32 values (a sum that
    cancelled down to 24 significant bits): there the fused value can round the other way, by one ulp."""
    from toda_b200 import synth
    rng = np.random.default_rng(0)
    n, ties = 0, 0
    for cfg, i in (("nus_0075", 0), ("nus_0075", 1), ("waymo_010", 0)):
        xyz = np.ascontiguousarray(synth.make_frame(cfg, i)[:, :3])
        u = rng.random()
        for w in (0.0, u * 2 * np.pi / 3, (u + 1) * 2 * np.pi / 3, np.pi / 2):
            got, ref = RP.rotate_xyz(xyz, w), np.dot(xyz, RP.rot_mat(w)).astype(F32)
            n += xyz.size
            rows, cols = np.nonzero(got.view(np.int32) != ref.view(np.int32))
            R, d = RP.rot_mat(w), xyz[rows].astype(np.float64)
            exact = (d[:, 0] * R[0, cols] + d[:, 1] * R[1, cols]) + d[:, 2] * R[2, cols]
            g, r = got[rows, cols], ref[rows, cols]
            assert np.all(np.abs(g.view(np.int32).astype(np.int64) - r.view(np.int32).astype(np.int64)) == 1), (cfg, i, w)
            assert np.all(exact == (g.astype(np.float64) + r.astype(np.float64)) / 2), (cfg, i, w)   # an exact tie
            ties += rows.size
    assert n > 3_000_000 and ties <= 3, ties


@pytest.mark.parametrize("cols", [7, 9, 10])
def test_plugin_candidate_boxes_equal_the_restatement(cols):
    """The host side of pcdet_plugin.processor.rotate_paste_points (step 1) computes the restatement's candidates."""
    from toda_b200.pcdet_plugin.processor import rotate_boxes_about_z, rotation_cos_sin
    rng = np.random.default_rng(cols)
    boxes = np.concatenate([rng.uniform(-50, 50, (200, 3)), rng.uniform(0.5, 5, (200, 3)), rng.uniform(-np.pi, np.pi, (200, 1)),
                            rng.normal(0, 2, (200, cols - 7))], 1)
    for dtype in (np.float32, np.float64):
        angles = [0.0, rng.random() * 2 * np.pi / 3, 2.5, -1.0]
        for cs, w in zip(rotation_cos_sin(angles), angles):
            assert cs.tolist() == [np.cos(w), np.sin(w)]
            assert _bits_equal(rotate_boxes_about_z(boxes.astype(dtype), cs, w), RP.rotate_boxes(boxes.astype(dtype), w))
