"""PolarMix rotate-pasting on the GPU (K0 rotate-paste kernels, ops.rotate_paste, pcdet_plugin.processor.rotate_paste_points)
against the restatement in tests/rotate_paste_oracle.py.  Points must be bit-identical; offsets, accepted flags, boxes
(in their dtype) and names must be equal."""
import numpy as np
import pytest
import torch

from oracle import points as OP
from tests import parity_utils as PU
from tests import rotate_paste_oracle as RP

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32 = np.float32
CLASSES = np.array(["car", "truck", "bus", "pedestrian", "bicycle"])


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, F32), np.ascontiguousarray(b, F32)
    return a.shape == b.shape and bool(((a.view(np.int32) == b.view(np.int32)) | (np.isnan(a) & np.isnan(b))).all())


def _boxes(rng, centres, cols, dtype=F32):
    """Car-sized boxes around the given (m, 3) centres, random headings, velocities (and a class column) after the 7."""
    m = centres.shape[0]
    size = np.array([4.5, 1.9, 1.6]) * rng.uniform(0.7, 1.3, (m, 3))
    extra = [rng.normal(0, 2, (m, 2))] if cols >= 9 else []
    extra += [rng.integers(1, 6, (m, 1)).astype(np.float64)] if cols == 10 else []
    return np.concatenate([centres, size, rng.uniform(-np.pi, np.pi, (m, 1))] + extra, 1).astype(dtype)


def _on_points(rng, frame, m, cols):
    """m instance boxes centred on points of the frame, so that they hold points."""
    if frame.shape[0] == 0:
        return _boxes(rng, rng.uniform(-40, 40, (m, 3)), cols)
    return _boxes(rng, frame[rng.integers(0, frame.shape[0], m), :3].astype(np.float64), cols)


def _names(rng, m):
    return CLASSES[rng.integers(0, len(CLASSES), m)]


def _batch(frames, x_col):
    offs = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)
    cols = [np.concatenate([np.full((f.shape[0], 1), b, F32), f], 1) if x_col else f for b, f in enumerate(frames)]
    return _t(np.concatenate(cols)), _t(offs)


def _polarmix_angles(rng):
    u = rng.random()
    return [0.0, u * 2 * np.pi / 3, (u + 1) * 2 * np.pi / 3]


def _oracle(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles):
    return [RP.rotate_paste_frame(d, s, g, gn, m, mn, a)
            for d, s, g, gn, m, mn, a in zip(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles)]


def _run(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles, x_col, same=False):
    from toda_b200 import ops
    from toda_b200.pcdet_plugin.processor import rotate_boxes_about_z, rotate_paste_points, rotation_cos_sin
    dst, dst_off = _batch(dst_frames, x_col)
    src, src_off = (dst, dst_off) if same else _batch(src_frames, x_col)
    got = rotate_paste_points(dst, dst_off, src, src_off, gt, gt_names, inst, inst_names, angles, x_col=x_col)
    rot = [rotation_cos_sin(a) for a in angles]
    cands = [np.concatenate([rotate_boxes_about_z(m, cs, w) for cs, w in zip(r, a)]) if len(a) else np.zeros((0, m.shape[1]), F32)
             for m, r, a in zip(inst, rot, angles)]
    pts, offs, acc = ops.rotate_paste(dst, dst_off, src, src_off, gt, inst, cands, rot, x_col=x_col)
    assert torch.equal(pts, got[0]) and torch.equal(offs, got[1])           # a second call gives the same bits
    return got, acc


def _compare(got, acc, want, x_col):
    pts, offs = got[0].cpu().numpy(), got[1].cpu().numpy()
    assert offs[0] == 0 and offs[-1] == pts.shape[0]
    assert np.array_equal(acc, np.concatenate([w[3] for w in want]))
    for b, (p, gb, nm, _) in enumerate(want):
        rows = pts[offs[b]:offs[b + 1]]
        if x_col:
            assert np.all(rows[:, 0] == b)
        assert _bits_equal(rows[:, x_col:], p), f"frame {b}: points differ"
        assert got[2][b].dtype == gb.dtype and _bits_equal(got[2][b], gb), f"frame {b}: boxes differ"
        assert list(got[3][b].astype(str)) == list(nm.astype(str)), f"frame {b}: names differ"


@pytest.fixture(scope="module")
def frames():
    from toda_b200 import synth
    return {cfg: [synth.make_frame(cfg, i) for i in range(8)] for cfg in ("nus_0075", "waymo_010")}


@pytest.mark.parametrize("same", [True, False])
@pytest.mark.parametrize("cols", [7, 9])
@pytest.mark.parametrize("x_col", [0, 1])
@pytest.mark.parametrize("cfg", ["nus_0075", "waymo_010"])
def test_full_frames_match_the_restatement(frames, cfg, x_col, cols, same):
    rng = np.random.default_rng([x_col, cols, int(same), len(cfg)])
    dst_frames = frames[cfg][:4]
    src_frames = dst_frames if same else frames[cfg][4:]
    gt = [_on_points(rng, f, 30, cols) for f in dst_frames]
    inst = [_on_points(rng, f, 40, cols) for f in src_frames]
    gt_names, inst_names = [_names(rng, 30) for _ in gt], [_names(rng, 40) for _ in inst]
    angles = [_polarmix_angles(rng) for _ in dst_frames]
    want = _oracle(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles)
    got, acc = _run(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles, x_col, same)
    _compare(got, acc, want, x_col)
    pasted = sum(w[0].shape[0] - d.shape[0] for w, d in zip(want, dst_frames))
    assert acc.sum() > 50 and (~acc).sum() > 0 and pasted > 10000, (acc.sum(), pasted)


def test_edge_frames():
    """An empty destination frame, an empty source frame, a frame without instance boxes, a frame whose candidates all
    collide with a destination box, a frame without angles, and a box with 10 columns in float64."""
    from toda_b200 import synth
    rng = np.random.default_rng(3)
    full = synth.make_frame("nus_0075", 2)
    other = synth.make_frame("nus_0075", 3)
    cover = np.array([[0, 0, 0, 500, 500, 20, 0, 0, 0, 1]], np.float64)
    dst_frames = [full[:0], full[:40000], full[40000:90000], full[90000:150000], full[150000:], full[:10]]
    src_frames = [other[:50000], other[:0], other[50000:90000], other[90000:], other[:30000], other[30000:]]
    inst = [_on_points(rng, s, m, 10) for s, m in zip(src_frames, (12, 7, 0, 20, 15, 25))]
    gt = [_boxes(rng, rng.uniform(-40, 40, (m, 3)), 10, np.float64) for m in (0, 5, 5, 0, 10, 3)]
    gt[3] = cover
    gt_names = [_names(rng, g.shape[0]) for g in gt]
    inst_names = [_names(rng, m.shape[0]) for m in inst]
    angles = [_polarmix_angles(rng), [0.0, 1.0], [0.5], [0.0, 2.0, 4.0], [], [0.0, 0.7, 1.9, 3.1]]
    for x_col in (0, 1):
        want = _oracle(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles)
        assert want[1][3].any() and want[1][0].shape[0] == 40000             # boxes pasted with zero rows
        assert not want[3][3].any() and want[3][3].shape == (60,)            # every candidate hits the cover box
        got, acc = _run(dst_frames, src_frames, gt, gt_names, inst, inst_names, angles, x_col)
        _compare(got, acc, want, x_col)
    # every source frame empty, a single frame, no instance box anywhere
    for s, m in ((full[:0], 5), (full, 0)):
        args = ([np.zeros((0, 7), F32)], [_names(rng, 0)], [_on_points(rng, full, m, 7)], [_names(rng, m)], [[0.0, 1.0]])
        want = _oracle([other], [s], *args)
        got, acc = _run([other], [s], *args, 1)
        _compare(got, acc, want, 1)


def test_limits_and_argument_errors():
    from toda_b200 import ops
    from toda_b200.pcdet_plugin.processor import rotate_paste_points
    pts = _t(np.zeros((4, 5), F32))
    off1 = _t(np.array([0, 4], np.int32))
    box = np.zeros((0, 7), F32)

    def call(n_frames=1, n_angles=1, n_inst=1, src=pts, x_col=0):
        off = _t(np.array([0, 4] + [4] * (n_frames - 1), np.int32))
        inst = [np.zeros((n_inst, 7), F32)] * n_frames
        rot = [np.tile([[1.0, 0.0]], (n_angles, 1))] * n_frames
        cand = [np.zeros((n_angles * n_inst, 7), F32)] * n_frames
        return ops.rotate_paste(pts, off, src, off, [box] * n_frames, inst, cand, rot, x_col=x_col)
    with pytest.raises(ValueError, match="at most 64"):
        call(n_frames=65)
    with pytest.raises(ValueError, match="17 angles"):
        call(n_angles=17)
    with pytest.raises(ValueError, match="1025 candidates"):
        call(n_angles=5, n_inst=205)
    with pytest.raises(ValueError, match="1025 instance boxes"):
        call(n_angles=0, n_inst=1025)
    with pytest.raises(ValueError, match="columns"):
        call(src=_t(np.zeros((4, 6), F32)))
    with pytest.raises(ValueError, match="stride"):
        ops.rotate_paste(_t(np.zeros((4, 3), F32)), off1, _t(np.zeros((4, 3), F32)), off1, [box], [box], [box],
                         [np.zeros((0, 2))], x_col=1)
    with pytest.raises(ValueError, match="columns"):
        rotate_paste_points(pts, off1, pts, off1, [box], [_names(np.random.default_rng(0), 0)], [np.zeros((1, 9), F32)],
                            [CLASSES[:1]], [[0.0]])
    out, offs, _ = call(n_angles=16, n_inst=64)                            # at the limits: 16 angles, 1024 candidates
    assert offs.tolist() == [0, out.shape[0]]
    # the library reports the same limits itself
    L, C = ops._C.lib(), ops._C
    alloc = C.ALLOC_FN(lambda rows, ctx: None)

    def raw(batch, counts, inst_off):
        return L.toda_rotate_paste(None, 0, None, None, 0, None, 5, 0, batch, None, C.ints([0] * (batch + 1)), None,
                                   C.ints(inst_off), None, None, C.ints(counts), None, alloc, None, None, None, 0, None)
    assert raw(65, [0] * 65, [0] * 66) == -4 and b"batch 65" in L.toda_last_error()
    assert raw(1, [17], [0, 1]) == -4 and b"17 angles" in L.toda_last_error()
    assert raw(1, [1], [0, 1025]) == -4 and b"1025 candidates" in L.toda_last_error()
    assert raw(1, [1], [0, 1]) == -1 and b"null" in L.toda_last_error()


def test_polar_swap_then_rotate_paste_then_voxelize():
    """polar_swap_points -> rotate_paste_points -> collate -> range mask -> MeanVFE.voxelize equals the oracle chain
    through the oracle voxelizer."""
    import toda_b200.pcdet_plugin as P
    from toda_b200 import synth
    from toda_b200.pcdet_plugin.processor import PointPreprocessor, collate_points, polar_swap_points, rotate_paste_points
    cfg = synth.CONFIGS["nus_0075"]
    pcr, vs = cfg["pc_range"], cfg["voxel_size"]
    rng = np.random.default_rng(11)
    pt1 = [synth.make_frame("nus_0075", i) for i in range(3)]
    pt2 = [synth.make_frame("waymo_010", i)[:, :5] for i in range(3)]
    sectors = [sorted(rng.uniform(-np.pi, np.pi, 2)) for _ in pt1]
    swapped = [OP.polar_swap_points(a, b, s, e) for a, b, (s, e) in zip(pt1, pt2, sectors)]
    gt = [_on_points(rng, f, 20, 9) for f in swapped]
    inst = [_on_points(rng, f, 30, 9) for f in pt2]
    gt_names, inst_names = [_names(rng, 20) for _ in gt], [_names(rng, 30) for _ in inst]
    angles = [_polarmix_angles(rng) for _ in pt1]
    want = _oracle(swapped, pt2, gt, gt_names, inst, inst_names, angles)

    dev_swapped = [polar_swap_points(_t(a), _t(b), s, e) for a, b, (s, e) in zip(pt1, pt2, sectors)]
    dst = torch.cat(dev_swapped)
    dst_off = _t(np.cumsum([0] + [x.shape[0] for x in dev_swapped]).astype(np.int32))
    src, src_off = _batch(pt2, 0)
    pts, offs, boxes, names = rotate_paste_points(dst, dst_off, src, src_off, gt, gt_names, inst, inst_names, angles)
    assert all(_bits_equal(b, w[1]) for b, w in zip(boxes, want))
    bd = {"points": collate_points(pts, offs), "point_frame_offsets": offs, "batch_size": len(pt1)}
    assert _bits_equal(bd["points"].cpu().numpy()[:, 1:], np.concatenate([w[0] for w in want]))
    # rotated copies can leave the range: the reference masks after the augmentations, before voxelization
    want = [OP.mask_points_outside_range(w[0], pcr) for w in want]
    pp = PointPreprocessor([PU.Cfg(NAME="mask_points_and_boxes_outside_range", REMOVE_OUTSIDE_BOXES=True),
                            PU.Cfg(NAME="transform_points_to_voxels_placeholder", VOXEL_SIZE=vs)], pcr, training=True,
                           num_point_features=5)
    bd = pp.forward(bd)
    assert _bits_equal(bd["points"].cpu().numpy(), OP.collate_points(want))
    vfe = P.MeanVFE(PU.Cfg(MAX_POINTS_PER_VOXEL=cfg["max_points"], MAX_NUMBER_OF_VOXELS=cfg["max_voxels"]), 5, voxel_size=vs,
                    point_cloud_range=pcr, grid_size=pp.grid_size).to(DEV).train()
    bd = vfe.voxelize(bd)
    coords = bd["voxel_coords"].cpu().numpy()
    counts = np.bincount(coords[:, 0], minlength=len(pt1)).tolist()
    got = (bd["voxels"].cpu().numpy(), coords, bd["voxel_num_points"].cpu().numpy(), np.array(counts + [sum(counts)]))
    ref = PU.oracle_voxelize_batch(want, pcr, vs, cfg["max_points"], cfg["max_voxels"]["train"])
    PU.assert_voxels_equal(got, ref, exact_order=False)
