"""Restatement of pcdet's DynamicMeanVFE.forward (OpenPCDet v0.5.2, pcdet/models/backbones_3d/vfe/dynamic_mean_vfe.py)
in numpy float32, for the tests.  No reference checkout is available; this is the pin.

    c      = floor((points[:, 1:4] - pc_range[0:3]) / voxel_size)     float32, per axis
    kept   = 0 <= c < grid_size on all three axes                        (NaN coordinates fail the test: dropped)
    key    = ((b * X + cx) * Y + cy) * Z + cz                            int64 (the reference's int32 key wraps)
    voxels = np.unique(key)                                               rows in ascending key order = (b, x, y, z)
    mean   = (float32 sum of points[i, 1:] over the voxel's points, added in ascending i from 0) / float32(count)

The sum is np.add.at into float32 zeros, which adds in index order (torch_scatter's CPU scatter_mean).
"""
import numpy as np


def dynamic_mean_vfe(points, batch_size, pc_range, voxel_size, grid_size):
    """points (N, 1+F) [b, x, y, z, ...] -> features (V, F) float32, coords (V, 4) int32 [b, z, y, x] and counts (B+1,)
    int32 (per-frame V_b, then V).  Rows in the reference's order (ascending (b, x, y, z) key)."""
    pts = np.ascontiguousarray(points, dtype=np.float32)
    n_feat = pts.shape[1] - 1
    lo = np.asarray(pc_range, dtype=np.float32)[0:3]
    vs = np.asarray(voxel_size, dtype=np.float32)
    grid = np.asarray(grid_size, dtype=np.int64)
    with np.errstate(invalid="ignore"):
        q = np.floor((pts[:, 1:4] - lo) / vs)
        keep = np.all((q >= 0) & (q < grid), axis=1)
    c = q[keep].astype(np.int64)
    b = pts[keep, 0].astype(np.int64)
    nx, ny, nz = (int(g) for g in grid)
    key = ((b * nx + c[:, 0]) * ny + c[:, 1]) * nz + c[:, 2]
    uniq, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
    sums = np.zeros((uniq.size, n_feat), np.float32)
    np.add.at(sums, inv.reshape(-1), pts[keep, 1:])
    features = sums / cnt.astype(np.float32)[:, None]
    ub, rem = np.divmod(uniq, nx * ny * nz)
    ux, rem = np.divmod(rem, ny * nz)
    uy, uz = np.divmod(rem, nz)
    coords = np.stack([ub, uz, uy, ux], axis=1).astype(np.int32)
    per_frame = np.bincount(ub, minlength=batch_size)[:batch_size]
    counts = np.concatenate([per_frame, [uniq.size]]).astype(np.int32)
    return features.astype(np.float32), coords, counts


def canonical(features, coords):
    """Rows sorted by (b, z, y, x), the order the GPU path emits."""
    o = np.lexsort((coords[:, 3], coords[:, 2], coords[:, 1], coords[:, 0]))
    return features[o], coords[o]
