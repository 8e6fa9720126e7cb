"""The DynamicMeanVFE restatement (tests/dynamic_vfe_oracle.py) on hand-derived cases, and tied to the hard-voxelizer
oracle that the goldens pin: with no cap binding, hard voxelization followed by MeanVFE is the same computation."""
import numpy as np

from oracle import voxelize as OV
from tests import dynamic_vfe_oracle as DV

PCR = [0.0, 0.0, 0.0, 4.0, 4.0, 4.0]
VS = [1.0, 1.0, 1.0]
GRID = [4, 4, 4]
TINY = np.float32(2.0 ** -24)


def _run(rows, batch_size=1):
    return DV.dynamic_mean_vfe(np.asarray(rows, np.float32), batch_size, PCR, VS, GRID)


def test_two_points_in_one_voxel_average():
    f, c, n = _run([[0, 0.5, 0.5, 0.5, 1.0], [0, 0.25, 0.75, 0.5, 3.0]])
    assert c.tolist() == [[0, 0, 0, 0]] and n.tolist() == [1, 1]
    assert f.tolist() == [[0.375, 0.625, 0.5, 2.0]]


def test_three_point_mean_adds_in_ascending_point_order():
    # (2^-24 + 2^-24) + 1 = 1 + 2^-23, while 1 + 2^-24 rounds back to 1: only the ascending order gives the first
    f, _, _ = _run([[0, 1.5, 1.5, 1.5, TINY], [0, 1.5, 1.5, 1.5, TINY], [0, 1.5, 1.5, 1.5, 1.0]])
    want = np.float32(np.float32(1.0) + np.float32(2.0 ** -23)) / np.float32(3)
    other = np.float32(1.0) / np.float32(3)
    assert want != other
    assert f[0, 3] == want


def test_range_edges_and_z():
    rows = [[0, 0.0, 0.0, 0.0, 1.0],        # exactly on lo: kept, voxel (0, 0, 0)
            [0, 4.0, 1.0, 1.0, 2.0],        # quotient exactly grid on x: dropped
            [0, 1.0, 1.0, 4.5, 3.0],        # x, y inside, z above the range: dropped
            [0, 1.0, 1.0, -0.5, 4.0],       # z below the range: dropped
            [0, 3.999, 3.999, 3.999, 5.0]]  # last cell: kept
    f, c, n = _run(rows)
    assert c.tolist() == [[0, 0, 0, 0], [0, 3, 3, 3]]
    assert f[:, 3].tolist() == [1.0, 5.0] and n.tolist() == [2, 2]


def test_nan_rows_are_dropped():
    nan = np.nan
    f, c, n = _run([[0, nan, 1.5, 1.5, 7.0], [0, 1.5, 1.5, 1.5, 1.0], [0, 1.5, nan, 1.5, 9.0], [0, 1.5, 1.5, nan, 9.0]])
    assert c.tolist() == [[0, 1, 1, 1]] and f[0, 3] == 1.0 and n.tolist() == [1, 1]


def test_rows_follow_the_reference_key_order():
    # voxel A at x=0, z=3 and voxel B at x=3, z=0: the (b, x, y, z) key puts A first, canonical (b, z, y, x) order B
    f, c, _ = _run([[0, 3.5, 0.5, 0.5, 2.0], [0, 0.5, 0.5, 3.5, 1.0]])
    assert c.tolist() == [[0, 3, 0, 0], [0, 0, 0, 3]]
    assert f[:, 3].tolist() == [1.0, 2.0]
    fc, cc = DV.canonical(f, c)
    assert cc.tolist() == [[0, 0, 0, 3], [0, 3, 0, 0]] and fc[:, 3].tolist() == [2.0, 1.0]


def test_batch_index_above_frame_zero():
    f, c, n = _run([[2, 0.5, 1.5, 2.5, 1.0], [2, 0.5, 1.5, 2.5, 2.0]], batch_size=3)
    assert c.tolist() == [[2, 2, 1, 0]] and n.tolist() == [0, 0, 1, 1] and f[0, 3] == 1.5


def test_restatement_equals_hard_voxelizer_without_caps():
    from toda_b200 import synth
    cfg = synth.CONFIGS["nus_0075"]
    pcr = [-6.0, -6.0, -5.0, 6.0, 6.0, 3.0]
    frames = []
    for i in range(2):
        fr = synth.make_frame("nus_0075", i)
        frames.append(fr[(np.abs(fr[:, 0]) < 7.0) & (np.abs(fr[:, 1]) < 7.0)])
    collated = np.concatenate([np.pad(fr, ((0, 0), (1, 0)), constant_values=b) for b, fr in enumerate(frames)])
    grid = OV.grid_size_xyz(pcr, cfg["voxel_size"])
    f, c, n = DV.dynamic_mean_vfe(collated, 2, pcr, cfg["voxel_size"], grid)
    f, c = DV.canonical(f, c)
    assert n[2] > 1000 and np.bincount(c[:, 0], minlength=2).tolist() == n[:2].tolist()
    want_f, want_c = [], []
    for b, fr in enumerate(frames):
        # K = the largest number of points any cell holds (out-of-range cells included), so no voxel is cut
        k = int(np.unique(np.floor((fr[:, :3] - np.float32(pcr[:3])) / np.float32(cfg["voxel_size"])), axis=0,
                          return_counts=True)[1].max())
        g = OV.Point2VoxelCPU3d(cfg["voxel_size"], pcr, fr.shape[1], k, fr.shape[0])
        v, cz, num = [t.numpy() for t in g.point_to_voxel(OV.from_numpy(fr))]
        want_f.append(OV.mean_vfe(v, num))
        want_c.append(np.pad(cz, ((0, 0), (1, 0)), constant_values=b))
    wf, wc = DV.canonical(np.concatenate(want_f), np.concatenate(want_c).astype(np.int32))
    assert np.array_equal(c, wc)
    assert np.array_equal(f.view(np.uint32), wf.view(np.uint32))
