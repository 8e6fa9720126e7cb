"""The world-augmentation restatement (tests/world_aug_oracle.py, restated from OpenPCDet v0.5.2) against hand-derived
cases, the torch CPU matmul dispatch that the device kernel reproduces, and the plugin's draw order -- runs on CPU."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU
from tests import world_aug_oracle as WA

F32 = np.float32
STEPS = [PU.Cfg(NAME="random_world_flip", ALONG_AXIS_LIST=["x", "y"]),
         PU.Cfg(NAME="random_world_rotation", WORLD_ROT_ANGLE=[-0.78539816, 0.78539816]),
         PU.Cfg(NAME="random_world_scaling", WORLD_SCALE_RANGE=[0.95, 1.05])]


def _frame(n, seed, f=5):
    return (np.random.default_rng(seed).standard_normal((n, f)) * 30).astype(F32)


def _cos_sin(angle):
    a = torch.from_numpy(np.array([angle])).float()
    return F32(torch.cos(a).item()), F32(torch.sin(a).item())


def _unfused(p, c, s):
    """ATen's naive bmm loop: acc = 0; acc += v[k] * R[k][j], every product and sum rounded to float32."""
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    zero, one = F32(0), F32(1)
    return np.stack([((zero + x * c) + y * -s) + z * zero,
                     ((zero + x * s) + y * c) + z * zero,
                     ((zero + x * zero) + y * zero) + z * one], 1)


def _fmaf(a, b, c):
    """float32 fma(a, b, c), exactly: a*b is exact in float64; the float64 sum's rounding error (TwoSum) decides the one
    case in which rounding twice differs from rounding once, a float64 sum that lands on a float32 midpoint."""
    a, b, c = (np.asarray(v, np.float64) for v in (a, b, c))
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    r = s.astype(F32)
    r64 = r.astype(np.float64)
    other = np.nextafter(r, np.where(s > r64, F32(np.inf), F32(-np.inf))).astype(F32)
    mid = (r64 != s) & (other.astype(np.float64) - s == s - r64)
    fix = mid & (err != 0) & (np.sign(err) == np.sign(s - r64))
    return np.where(fix, other, r)


def _fused(p, c, s):
    """The BLAS path: acc = fma(v[k], R[k][j], acc) from acc = 0."""
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    zero, one = F32(0), F32(1)
    return np.stack([_fmaf(z, zero, _fmaf(y, -s, _fmaf(x, c, zero))),
                     _fmaf(z, zero, _fmaf(y, c, _fmaf(x, s, zero))),
                     _fmaf(z, one, _fmaf(y, zero, _fmaf(x, zero, zero)))], 1)


def test_flips_are_involutions():
    p = _frame(100, 1)
    boxes = _frame(7, 2, 9)
    for flip in (WA.random_flip_along_x, WA.random_flip_along_y):
        b1, p1 = flip(boxes.copy(), p.copy(), True)
        assert not np.array_equal(p1, p)
        b2, p2 = flip(b1, p1, True)
        assert np.array_equal(p2, p) and np.array_equal(b2[:, [0, 1, 7, 8]], boxes[:, [0, 1, 7, 8]])
        b3, p3 = flip(boxes.copy(), p.copy(), False)
        assert np.array_equal(p3, p) and np.array_equal(b3, boxes)
    _, p1 = WA.random_flip_along_x(boxes.copy(), p.copy(), True)
    assert np.array_equal(p1[:, 1], -p[:, 1]) and np.array_equal(np.delete(p1, 1, 1), np.delete(p, 1, 1))
    _, p1 = WA.random_flip_along_y(boxes.copy(), p.copy(), True)
    assert np.array_equal(p1[:, 0], -p[:, 0]) and np.array_equal(p1[:, 1:], p[:, 1:])


@pytest.mark.parametrize("n", [3, 44, 45, 5000])
def test_rotation_by_zero_is_the_identity(n):
    p = _frame(n, n)
    got = WA.rotate_points_along_z(p[np.newaxis], np.array([0.0]))[0]
    assert np.array_equal(got, p)


def test_quarter_turn_follows_the_reference_sign_convention():
    """xyz @ [[c, s, 0], [-s, c, 0], [0, 0, 1]]: (1, 0) goes to (c, s) and (0, 1) to (-s, c), i.e. counter-clockwise."""
    c, s = _cos_sin(np.pi / 2)
    p = np.array([[1, 0, 0, 9], [0, 1, 0, 9], [0, 0, 2, 9]], F32)
    got = WA.rotate_points_along_z(p[np.newaxis], np.array([np.pi / 2]))[0]
    assert np.array_equal(got[0, :2], [c, s]) and np.array_equal(got[1, :2], [-s, c])
    assert got[2, 2] == 2 and np.array_equal(got[:, 3], p[:, 3])
    assert abs(c) < 1e-7 and s == 1


def test_torch_matmul_dispatch_is_pinned():
    """The kernel picks the rounding of the rotation from the frame's row count, as torch 2.x's CPU matmul does for a
    (1, N, 3) x (1, 3, 3) product: ATen's naive bmm loop (unfused) while 3 * N * 3 < 400, i.e. N <= 44, and the BLAS
    kernel (a chain of fmas) from N = 45.  If this fails, the host's torch rounds the reference's rotation differently
    and the device kernel (toda_points_world_transform) must follow it."""
    angle = 0.6172
    c, s = _cos_sin(angle)
    for seed in range(20):
        p = _frame(44, seed)
        got = WA.rotate_points_along_z(p[np.newaxis], np.array([angle]))[0]
        assert np.array_equal(got[:, :3], _unfused(p, c, s)), f"N=44, seed {seed}: torch no longer uses the unfused naive loop"
    differs = 0
    for seed in range(20):
        p = _frame(45, seed)
        got = WA.rotate_points_along_z(p[np.newaxis], np.array([angle]))[0]
        assert np.array_equal(got[:, :3], _fused(p, c, s)), f"N=45, seed {seed}: torch no longer rounds as a chain of fmas"
        differs += int(not np.array_equal(got[:, :3], _unfused(p, c, s)))
    assert differs > 0, "the fused and unfused forms never disagreed: the check has no power"
    p = _frame(300000, 1)
    got = WA.rotate_points_along_z(p[np.newaxis], np.array([angle]))[0]
    assert np.array_equal(got[:, :3], _fused(p, c, s))


def test_scaling_multiplies_in_float32():
    p = _frame(50, 3)
    boxes = _frame(4, 4, 7).astype(np.float64)
    b, got = WA.global_scaling(boxes.copy(), p.copy(), 1.0123456789)
    assert got.dtype == F32 and np.array_equal(got[:, :3], p[:, :3] * F32(1.0123456789))
    assert np.array_equal(got[:, 3:], p[:, 3:]) and np.array_equal(b[:, :6], boxes[:, :6] * 1.0123456789)
    b, got = WA.global_scaling(boxes.copy(), p.copy(), None)
    assert np.array_equal(got, p) and np.array_equal(b, boxes)


def test_plugin_draws_follow_the_reference_order():
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    for steps in (STEPS, STEPS[::-1], [STEPS[1], STEPS[0]],
                  STEPS[:2] + [PU.Cfg(NAME="random_world_scaling", WORLD_SCALE_RANGE=[1.0, 1.0005])],
                  [PU.Cfg(NAME="random_world_rotation", WORLD_ROT_ANGLE=0.3)]):
        aug = DataAugmentor(steps)
        np.random.seed(1234)
        got = [[st.draw() for st in aug.data_augmentor_queue] for _ in range(5)]
        np.random.seed(1234)
        want = [WA.draw_world_augmentations(steps) for _ in range(5)]
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert len(g) == len(w)
            for a, b in zip(g, w):
                assert (a is None and b is None) or np.array_equal(np.asarray(a), np.asarray(b))


def test_plugin_boxes_match_the_oracle():
    """The host box path of the plugin (the reference's expressions) against the restatement, per frame."""
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor, _limit_period
    aug = DataAugmentor(STEPS)
    np.random.seed(5)
    for cols in (7, 9, 10):
        for dtype in (np.float32, np.float64):
            for m in (3, 44, 45, 60):
                boxes = _frame(m, m + cols, cols).astype(dtype)
                draws = [st.draw() for st in aug.data_augmentor_queue]
                got = boxes.copy()
                for st, d in zip(aug.data_augmentor_queue, draws):
                    got = st.boxes(got, d)
                got[:, 6] = _limit_period(got[:, 6], offset=0.5, period=2 * np.pi)
                _, want = WA.world_augment(np.zeros((1, 4), F32), boxes, STEPS, draws)
                assert got.dtype == dtype and np.array_equal(got, want), (cols, dtype, m)


def test_augmentor_config_protocol():
    from toda_b200.pcdet_plugin.augmentor import DataAugmentor
    cfg = PU.Cfg(DISABLE_AUG_LIST=["placeholder"], AUG_CONFIG_LIST=[PU.Cfg(NAME="gt_sampling")] + STEPS)
    with pytest.raises(NotImplementedError, match="gt_sampling"):
        DataAugmentor(cfg)
    assert len(DataAugmentor(cfg, host_steps=("gt_sampling",)).data_augmentor_queue) == 3
    cfg = PU.Cfg(DISABLE_AUG_LIST=["gt_sampling", "random_world_flip"], AUG_CONFIG_LIST=[PU.Cfg(NAME="gt_sampling")] + STEPS)
    assert [s.name for s in DataAugmentor(cfg).data_augmentor_queue] == ["random_world_rotation", "random_world_scaling"]
    with pytest.raises(NotImplementedError, match="random_local_rotation"):
        DataAugmentor([PU.Cfg(NAME="random_local_rotation", LOCAL_ROT_ANGLE=[-0.1, 0.1])])
