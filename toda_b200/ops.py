"""Host-side (PyTorch) wrappers over the C ABI: tensors in, tensors out, autograd where the
reference differentiates through the op.  PyTorch is plumbing here (device memory, streams, autograd
graph); every device-side computation is a kernel of libtoda_b200.so.  No CPU fallback.
"""
import ctypes
import weakref
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _C

ORDER_FIRST_APPEARANCE = 0
ORDER_CANONICAL = 1
CONV_FP32 = 0
CONV_BF16 = 1
CONV_BF16X3 = 2      # split-bf16, three tensor-core launches per product: fp32-class accuracy (csrc/conv_x3.cu)

# launches of this library's kernels since the last reset (bench.py reports it as gpu_launches): counted inside the
# library, at every launch site (toda_launch_count)
_launch_base = 0


def launches():
    return int(_C.lib().toda_launch_count()) - _launch_base


def reset_launches():
    global _launch_base
    _launch_base = int(_C.lib().toda_launch_count())



# optional per-call device timing (bench.py's roofline pass): list of (name, meta, start_event, end_event)
_prof = None


def profile_begin():
    global _prof
    _prof = []


def profile_end():
    """-> list of dicts {name, ms, **meta}; synchronises."""
    global _prof
    rec, _prof = _prof, None
    torch.cuda.synchronize()
    return [dict(name=n, ms=a.elapsed_time(b), **m) for (n, m, a, b) in rec]


class _Timed:
    def __init__(self, name, meta):
        self.name, self.meta = name, meta

    def __enter__(self):
        self.a = torch.cuda.Event(enable_timing=True)
        self.a.record()
        return self

    def __exit__(self, *exc):
        b = torch.cuda.Event(enable_timing=True)
        b.record()
        _prof.append((self.name, self.meta, self.a, b))
        return False


class _NoTimer:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NO_TIMER = _NoTimer()


def _timed(name, **meta):
    """Context manager around one C-ABI call: records CUDA events only while a profile pass is active."""
    return _Timed(name, meta) if _prof is not None else _NO_TIMER


_raw_stream = torch._C._cuda_getCurrentRawStream     # (device index) -> cudaStream_t as int: ~0.2 us, torch.cuda.current_stream() ~8 us


def _stream_id(device=None):
    return _raw_stream(torch.cuda.current_device() if device is None or device.index is None else device.index)


def _stream():
    return ctypes.c_void_p(_raw_stream(torch.cuda.current_device()))


def _p(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _need(t, dtype, name):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (toda_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    return t


_workspaces = {}


def _workspace(tag, nbytes, device, zero=False):
    """Grow-only cached scratch buffers (caller-owned memory in the ABI's terms).  One buffer per (tag, device, STREAM):
    the input pipeline runs the front of batch i+1 on a side stream while the main stream may still use the same tag, and
    a block must never be shared (or regrown, which frees the old block into another stream's pool) across streams."""
    key = (tag, device.index, _stream_id(device))
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = (torch.zeros if zero else torch.empty)(int(nbytes * 1.25) + 256, dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


# ------------------------------------------------------------------------------------------------
# K0 point-stream selection
# ------------------------------------------------------------------------------------------------
SELECT_RANGE_XY, SELECT_RECT_XY, SELECT_SECTOR, SELECT_BOXES = 0, 1, 2, 3
SELECT_MAX_BOXES = 96


def points_select(points, frame_offsets, mode, params, invert=False, add_batch_col=False, x_col=0, trim=True):
    """Order-preserving selection of point rows (numpy `points[mask]` for a whole batch of frames).

    points (N, stride) float32 CUDA; frame_offsets int32 (B+1) CUDA tensor or None.  mode / params: see
    include/toda_b200.h (range mask of common_utils.mask_points_by_range, cutmix rectangle, PolarMix sector).
    Returns (rows, offsets): rows (N', stride[+1]) and int32 offsets (B+1) (or (1,) = N' without frames).
    trim=True slices to N' (one host sync); trim=False returns the capacity-sized buffer.
    """
    points = _need(points, torch.float32, "points")
    assert points.dim() == 2
    n, stride = points.shape
    dev = points.device
    batch = 0
    if frame_offsets is not None:
        frame_offsets = _need(frame_offsets, torch.int32, "frame_offsets")
        batch = frame_offsets.numel() - 1
    L = _C.lib()
    ws = _workspace("select", L.toda_points_select_workspace_bytes(n), dev)
    out = torch.empty((n, stride + (1 if add_batch_col else 0)), dtype=torch.float32, device=dev)
    out_offsets = torch.empty((batch + 1,), dtype=torch.int32, device=dev)
    p = list(params) + [0.0] * (4 - len(params))
    with _timed("points_select", n=n, stride=stride, mode=int(mode)):
        _C.check(L.toda_points_select(_p(points), n, stride, int(x_col), _p(frame_offsets), batch, int(mode), _C.doubles(p),
                                      int(bool(invert)), int(bool(add_batch_col)), _p(out), _p(out_offsets), _p(ws),
                                      ws.numel(), _stream()), "toda_points_select")
    if trim:
        return out[:int(out_offsets[-1].item())], out_offsets
    return out, out_offsets


WORLD_FLIP_X, WORLD_FLIP_Y, WORLD_ROTATE, WORLD_SCALE = 0, 1, 2, 3
WORLD_MAX_STEPS = 4
WORLD_MAX_BATCH = 64


def points_world_transform(points, frame_offsets, steps, x_col=0):
    """The point side of pcdet's world augmentations (random_world_flip / _rotation / _scaling) for a batch of frames,
    bit-identical to the reference's float32 arithmetic (see include/toda_b200.h).  Returns a new (N, stride) tensor.

    points (N, stride) float32 CUDA with x, y, z at x_col..x_col+2; frame_offsets int32 (B+1) CUDA tensor or None (one
    frame).  steps: at most 4 (kind, per-frame values) pairs applied in order, one value per frame:
      WORLD_FLIP_X / WORLD_FLIP_Y  whether the flip is enabled
      WORLD_ROTATE                 (cos, sin) of the float32 angle as torch.cos / torch.sin give them
      WORLD_SCALE                  the scale factor (rounded to float32)
    """
    points = _need(points, torch.float32, "points")
    if points.dim() != 2:
        raise ValueError("points must be (N, stride)")
    n, stride = points.shape
    if not (0 <= x_col and x_col + 2 < stride <= 63):
        raise ValueError(f"points_world_transform: x, y, z at columns {x_col}..{x_col + 2} do not fit stride {stride} (<= 63)")
    batch = 1
    if frame_offsets is not None:
        frame_offsets = _need(frame_offsets, torch.int32, "frame_offsets")
        batch = frame_offsets.numel() - 1
        if not 1 <= batch <= WORLD_MAX_BATCH:
            raise ValueError(f"points_world_transform: batch {batch} outside [1, {WORLD_MAX_BATCH}]")
    if len(steps) > WORLD_MAX_STEPS:
        raise ValueError(f"points_world_transform: {len(steps)} steps (at most {WORLD_MAX_STEPS})")
    kinds, params = [], np.zeros((len(steps), batch, 2), np.float32)
    for s, (kind, values) in enumerate(steps):
        if kind not in (WORLD_FLIP_X, WORLD_FLIP_Y, WORLD_ROTATE, WORLD_SCALE):
            raise ValueError(f"points_world_transform: unknown step kind {kind!r}")
        v = np.asarray(values, dtype=np.float32).reshape(batch, -1)
        if v.shape[1] != (2 if kind == WORLD_ROTATE else 1):
            raise ValueError(f"points_world_transform: step {s} needs {2 if kind == WORLD_ROTATE else 1} value(s) per frame for "
                             f"{batch} frame(s), got {np.shape(values)}")
        kinds.append(int(kind))
        params[s, :, :v.shape[1]] = v
    out = torch.empty_like(points)
    with _timed("points_world_transform", n=n, stride=stride, steps=len(steps)):
        _C.check(_C.lib().toda_points_world_transform(_p(points), n, stride, int(x_col), _p(frame_offsets), batch, len(kinds),
                                                      _C.ints(kinds or [0]), _C.floats(params.reshape(-1).tolist() or [0.0]),
                                                      _p(out), _stream()), "toda_points_world_transform")
    return out


GTS_MAX_BATCH = 64
GTS_MAX_GROUPS = 16
GTS_MAX_SAMPLES_PER_FRAME = 1024


def gt_sampling_pack_boxes(boxes, extra_width=None):
    """(n, 7+) boxes -> float32 (n, 16) table of the device's box format (include/toda_b200.h), made by the library's host
    code: the first 7 columns cast to float32, libm cosf / sinf of the heading and of its negation, and the sizes
    enlarged by extra_width in float32."""
    b = np.ascontiguousarray(np.asarray(boxes)[:, :7], dtype=np.float32)
    out = np.zeros((b.shape[0], 16), np.float32)
    w = None if extra_width is None else np.ascontiguousarray(extra_width, dtype=np.float32)
    _C.check(_C.lib().toda_gt_sampling_pack_boxes(b.ctypes.data, b.shape[0], None if w is None else w.ctypes.data,
                                                  out.ctypes.data), "toda_gt_sampling_pack_boxes")
    return out


def gt_sampling(points, frame_offsets, gt_boxes, sampled_boxes, group_sizes, db_points, sample_rows, sample_centres,
                centres_f64, extra_width, x_col=0):
    """The device side of pcdet's gt_sampling for a batch of frames (collision test, scene-point removal, paste; see
    include/toda_b200.h).  One host-to-device copy of the box tables and one device-to-host copy of the accepted flags
    and the new frame offsets, which is the only host synchronisation.

    points (N, x_col + F) float32 CUDA, frame_offsets int32 (B+1) CUDA.  gt_boxes: B host arrays (M_b, 7+), each frame's
    unmasked gt boxes.  sampled_boxes (S, 7+) host, frame by frame and within a frame group by group; group_sizes (B, G)
    host ints.  db_points (R, F) float32 CUDA; sample_rows (S, 2) host: first row and row count of each sample's object
    points; sample_centres (S, 3) host: box3d_lidar[:3] of each sample (float64 values of the database's box dtype);
    centres_f64: the database stores float64 boxes.  extra_width: REMOVE_EXTRA_WIDTH.
    Returns (points, frame_offsets, accepted) with accepted a host bool array (S,).
    """
    points = _need(points, torch.float32, "points")
    frame_offsets = _need(frame_offsets, torch.int32, "frame_offsets")
    db_points = _need(db_points, torch.float32, "db_points")
    if points.dim() != 2 or db_points.dim() != 2:
        raise ValueError("gt_sampling: points and db_points must be 2-D")
    n, stride = points.shape
    feat = db_points.shape[1]
    batch = frame_offsets.numel() - 1
    if x_col not in (0, 1) or stride != x_col + feat:
        raise ValueError(f"gt_sampling: points have {stride} columns, the database {feat} features (x_col={x_col})")
    if not 1 <= batch <= GTS_MAX_BATCH or len(gt_boxes) != batch:
        raise ValueError(f"gt_sampling: {batch} frames and {len(gt_boxes)} gt_boxes arrays (at most {GTS_MAX_BATCH} frames)")
    group_sizes = np.asarray(group_sizes, np.int32).reshape(batch, -1)
    n_groups = group_sizes.shape[1]
    if not 1 <= n_groups <= GTS_MAX_GROUPS:
        raise ValueError(f"gt_sampling: {n_groups} sample groups (at most {GTS_MAX_GROUPS})")
    s = int(group_sizes.sum())
    if np.asarray(sampled_boxes).shape[0] != s or np.asarray(sample_rows).shape != (s, 2):
        raise ValueError(f"gt_sampling: the group sizes add up to {s} samples, the tables do not")
    exist = [gt_sampling_pack_boxes(g) for g in gt_boxes]
    exist_off = np.cumsum([0] + [e.shape[0] for e in exist]).astype(np.int32)
    rows = np.ascontiguousarray(sample_rows, dtype=np.int64)
    # one pinned staging buffer, one upload: gt box table | sample box table | sample rows | sample centres
    parts = [np.concatenate(exist) if exist_off[-1] else np.zeros((0, 16), np.float32),
             gt_sampling_pack_boxes(sampled_boxes, extra_width), rows, np.ascontiguousarray(sample_centres, dtype=np.float64)]
    offs, total = [], 0
    for p in parts:
        offs.append(total)
        total += (p.nbytes + 255) // 256 * 256
    staging = torch.empty(max(total, 256), dtype=torch.uint8, pin_memory=True)
    host = staging.numpy()
    for p, o in zip(parts, offs):
        host[o:o + p.nbytes] = np.frombuffer(p.tobytes(), np.uint8)
    dev = points.device
    tables = staging.to(dev, non_blocking=True)
    base = tables.data_ptr()
    L = _C.lib()
    ws = _workspace("gt_sampling", L.toda_gt_sampling_workspace_bytes(n, batch, s), dev)
    out = torch.empty((n + int(rows[:, 1].sum()), stride), dtype=torch.float32, device=dev)
    res = torch.empty((s + batch + 1,), dtype=torch.int32, device=dev)          # accepted flags | new frame offsets
    with _timed("gt_sampling", n=n, stride=stride, samples=s):
        _C.check(L.toda_gt_sampling(_p(points), n, stride, int(x_col), _p(frame_offsets), batch, ctypes.c_void_p(base + offs[0]),
                                    _C.ints(exist_off), ctypes.c_void_p(base + offs[1]), _C.ints(group_sizes.reshape(-1)),
                                    n_groups, _p(db_points), feat, ctypes.c_void_p(base + offs[2]),
                                    ctypes.c_void_p(base + offs[3]), int(bool(centres_f64)), _p(out), _p(res[s:]), _p(res),
                                    _p(ws), ws.numel(), _stream()), "toda_gt_sampling")
    back = res.cpu()
    new_offsets = res[s:]
    return out[:int(back[-1])], new_offsets, back[:s].numpy().astype(bool)


RP_MAX_BATCH = GTS_MAX_BATCH
RP_MAX_ANGLES = GTS_MAX_GROUPS
RP_MAX_CANDIDATES_PER_FRAME = GTS_MAX_SAMPLES_PER_FRAME


def rotate_paste(dst_points, dst_offsets, src_points, src_offsets, dst_boxes, inst_boxes, cand_boxes, rotations, x_col=0):
    """PolarMix's rotate-pasting for a batch of frames (collision test of the rotated instance copies and the paste of
    their points; see include/toda_b200.h).  One pinned host-to-device copy of the box tables and the angles' cos / sin,
    and one device-to-host copy of the accepted flags and the per-frame totals, which is the only host synchronisation.

    dst_points / src_points (N, x_col + F) float32 CUDA with the same columns (they may be the same tensor); dst_offsets /
    src_offsets int32 (B+1) CUDA.  Per frame, host arrays: dst_boxes[b] (E_b, 7+) destination boxes, inst_boxes[b]
    (M_b, 7+) instance boxes, rotations[b] (A_b, 2) float64 (cos w, sin w) of the A_b angles, cand_boxes[b] (A_b * M_b, 7+)
    the instance boxes rotated by each angle, angle by angle.  Returns (points, frame_offsets, accepted) with accepted a host bool array of the candidates,
    frame by frame.
    """
    dst_points = _need(dst_points, torch.float32, "dst_points")
    src_points = _need(src_points, torch.float32, "src_points")
    dst_offsets = _need(dst_offsets, torch.int32, "dst_offsets")
    src_offsets = _need(src_offsets, torch.int32, "src_offsets")
    if dst_points.dim() != 2 or src_points.dim() != 2:
        raise ValueError("rotate_paste: points must be (N, stride)")
    n_dst, stride = dst_points.shape
    if src_points.shape[1] != stride:
        raise ValueError(f"rotate_paste: source rows have {src_points.shape[1]} columns, destination rows {stride}")
    if x_col not in (0, 1) or not x_col + 3 <= stride <= 63:
        raise ValueError(f"rotate_paste: x, y, z at columns {x_col}..{x_col + 2} do not fit stride {stride} (<= 63)")
    batch = dst_offsets.numel() - 1
    if src_offsets.numel() - 1 != batch or not 1 <= batch <= RP_MAX_BATCH:
        raise ValueError(f"rotate_paste: {batch} destination and {src_offsets.numel() - 1} source frames "
                         f"(at most {RP_MAX_BATCH})")
    if not len(dst_boxes) == len(inst_boxes) == len(cand_boxes) == len(rotations) == batch:
        raise ValueError(f"rotate_paste: {batch} frames need {batch} box tables and rotation tables")
    rotations = [np.asarray(r, np.float64).reshape(-1, 2) for r in rotations]
    counts = np.array([r.shape[0] for r in rotations], np.int32)
    inst = [np.asarray(m).reshape(-1, np.shape(m)[-1]) for m in inst_boxes]
    for b, (a, m, c) in enumerate(zip(counts, inst, cand_boxes)):
        if a > RP_MAX_ANGLES:
            raise ValueError(f"rotate_paste: frame {b} has {a} angles (at most {RP_MAX_ANGLES})")
        if m.shape[0] > RP_MAX_CANDIDATES_PER_FRAME or a * m.shape[0] > RP_MAX_CANDIDATES_PER_FRAME:
            raise ValueError(f"rotate_paste: frame {b} has {m.shape[0]} instance boxes and {a * m.shape[0]} candidates "
                             f"(at most {RP_MAX_CANDIDATES_PER_FRAME} each)")
        if np.shape(c)[0] != a * m.shape[0]:
            raise ValueError(f"rotate_paste: frame {b} has {np.shape(c)[0]} candidate boxes, not {a} x {m.shape[0]}")
    packs = [[gt_sampling_pack_boxes(np.asarray(x).reshape(-1, np.shape(x)[-1])) for x in xs]
             for xs in (dst_boxes, inst, cand_boxes)]
    dst_off = np.cumsum([0] + [p.shape[0] for p in packs[0]]).astype(np.int32)
    inst_off = np.cumsum([0] + [p.shape[0] for p in packs[1]]).astype(np.int32)
    n_cand = sum(p.shape[0] for p in packs[2])
    # one pinned staging buffer, one upload: destination boxes | instance boxes | candidate boxes | cos / sin
    parts = [np.concatenate(p) for p in packs] + [np.concatenate(rotations)]
    offs, total = [], 0
    for p in parts:
        offs.append(total)
        total += (p.nbytes + 255) // 256 * 256
    staging = torch.empty(max(total, 256), dtype=torch.uint8, pin_memory=True)
    host = staging.numpy()
    for p, o in zip(parts, offs):
        host[o:o + p.nbytes] = np.frombuffer(p.tobytes(), np.uint8)
    dev = dst_points.device
    tables = staging.to(dev, non_blocking=True)
    base = tables.data_ptr()
    L = _C.lib()
    n_src = src_points.shape[0]
    ws = _workspace("rotate_paste", L.toda_rotate_paste_workspace_bytes(n_src, batch, max(p.shape[0] for p in packs[1]),
                                                                         n_cand), dev)
    result = torch.empty(n_cand + 2 * batch, dtype=torch.int32, pin_memory=True)
    out_offsets = torch.empty(batch + 1, dtype=torch.int32, device=dev)
    out = []

    def alloc(rows, _ctx):
        out.append(torch.empty((rows, stride), dtype=torch.float32, device=dev))
        return out[0].data_ptr() if rows else None
    alloc_fn = _C.ALLOC_FN(alloc)
    with _timed("rotate_paste", n_src=n_src, n_dst=n_dst, stride=stride, candidates=n_cand):
        _C.check(L.toda_rotate_paste(_p(src_points), n_src, _p(src_offsets), _p(dst_points), n_dst, _p(dst_offsets), stride,
                                     int(x_col), batch, ctypes.c_void_p(base + offs[0]), _C.ints(dst_off),
                                     ctypes.c_void_p(base + offs[1]), _C.ints(inst_off), ctypes.c_void_p(base + offs[2]),
                                     ctypes.c_void_p(base + offs[3]), _C.ints(counts), _p(result), alloc_fn, None,
                                     _p(out_offsets), _p(ws), ws.numel(), _stream()), "toda_rotate_paste")
    return out[0], out_offsets, result[:n_cand].numpy().astype(bool)


def gather_point_rows(points, rows):
    """out[i] = points[rows[i]] (numpy `points[idx]`): shuffle_points / mixup prefixes for a given index vector."""
    points = _need(points, torch.float32, "points")
    rows = _need(rows, torch.int32, "rows")
    n, c = rows.shape[0], points.shape[1]
    out = torch.empty((n, c), dtype=torch.float32, device=points.device)
    _C.check(_C.lib().toda_gather_rows(_p(points), _p(rows), n, c, _p(out), _stream()), "toda_gather_rows")
    return out


# ------------------------------------------------------------------------------------------------
# K1 voxelizer
# ------------------------------------------------------------------------------------------------
def grid_size_xyz(pc_range, voxel_size):
    """round((hi-lo)/vsize) -- pcdet/datasets/processor/data_processor.py L117-118."""
    r = np.asarray(pc_range, dtype=np.float64)
    return np.round((r[3:6] - r[0:3]) / np.asarray(voxel_size, dtype=np.float64)).astype(np.int64)


def voxelize(points, frame_offsets, pc_range, voxel_size, max_points, max_voxels, num_features=None, xyz_col=0,
             feat_col=0, order=ORDER_FIRST_APPEARANCE, grid=None, trim=True):
    """Hard voxelization of a batch of frames (replaces Point2VoxelCPU3d.point_to_voxel per frame +
    collate of dataset.py L171-178).

    points: (N, stride) float32 CUDA, frames back to back; frame_offsets: int32 (B+1) CUDA tensor or list.
    Returns voxels (V,K,F), coords (V,4)=[b,z,y,x] int32, num_points (V,) int32, counts (B+1,) int32
    (per-frame V_b, then V).  trim=True slices to V (one host sync); trim=False returns capacity-sized
    buffers and no sync.
    """
    points = _need(points, torch.float32, "points")
    assert points.dim() == 2
    n, stride = points.shape
    dev = points.device
    if not torch.is_tensor(frame_offsets):
        frame_offsets = torch.tensor(list(frame_offsets), dtype=torch.int32, device=dev)
    frame_offsets = _need(frame_offsets, torch.int32, "frame_offsets")
    batch = frame_offsets.numel() - 1
    f = int(num_features) if num_features is not None else stride - feat_col
    grid = grid_size_xyz(pc_range, voxel_size) if grid is None else np.asarray(grid)
    grid_c = _C.ints(grid)
    L = _C.lib()
    ws_bytes = L.toda_voxelize_workspace_bytes(n, batch, grid_c, max_points, max_voxels)
    if ws_bytes == 0:
        raise RuntimeError("toda_voxelize_workspace_bytes rejected the arguments")
    ws = _workspace("vox", ws_bytes, dev)
    cap = batch * max_voxels
    voxels = torch.empty((cap, max_points, f), dtype=torch.float32, device=dev)
    coords = torch.empty((cap, 4), dtype=torch.int32, device=dev)
    num = torch.empty((cap,), dtype=torch.int32, device=dev)
    counts = torch.empty((batch + 1,), dtype=torch.int32, device=dev)
    with _timed("voxelize", n_points=n, batch=batch, K=max_points, F=f):
        rc = L.toda_voxelize_hard(_p(points), n, stride, xyz_col, feat_col, f, _p(frame_offsets), batch,
                                  _C.floats(np.asarray(pc_range, dtype=np.float32)),
                                  _C.floats(np.asarray(voxel_size, dtype=np.float32)), grid_c, max_points, max_voxels,
                                  order, _p(voxels), _p(coords), _p(num), _p(counts), _p(ws), ws.numel(), _stream())
    _C.check(rc, "toda_voxelize_hard")
    if trim:
        v = int(counts[batch].item())
        return voxels[:v], coords[:v], num[:v], counts
    return voxels, coords, num, counts


def voxelize_dynamic(points, frame_offsets, pc_range, voxel_size, grid=None, xyz_col=1, feat_col=1):
    """Uncapped voxelization and per-voxel mean of a batch of frames (pcdet DynamicMeanVFE.forward, OpenPCDet v0.5.2,
    without torch_scatter).

    points: (N, stride) float32 CUDA, frames back to back, x,y,z at xyz_col..xyz_col+2; frame_offsets: int32 (B+1) CUDA
    tensor or list.  Every point inside [0, grid) on all three axes counts; the features are all columns from feat_col
    on, averaged over each voxel's points with an fp32 sum in ascending point order.  Returns features (V, F) float32,
    coords (V, 4) = [b, z, y, x] int32 in canonical order and counts (B+1,) int32 (per-frame V_b, then V).  One host
    sync (the voxel count).
    """
    if not torch.is_tensor(points):
        raise TypeError("voxelize_dynamic: points must be a torch tensor")
    points = _need(points, torch.float32, "points")
    if points.dim() != 2:
        raise ValueError(f"voxelize_dynamic: points must be (N, stride), got shape {tuple(points.shape)}")
    n, stride = points.shape
    dev = points.device
    if not torch.is_tensor(frame_offsets):
        frame_offsets = torch.tensor(list(frame_offsets), dtype=torch.int32, device=dev)
    frame_offsets = _need(frame_offsets, torch.int32, "frame_offsets")
    if frame_offsets.dim() != 1 or frame_offsets.numel() < 2:
        raise ValueError("voxelize_dynamic: frame_offsets must be a (B+1,) vector with B >= 1")
    batch = frame_offsets.numel() - 1
    xyz_col, feat_col = int(xyz_col), int(feat_col)
    if not (0 <= xyz_col and xyz_col + 3 <= stride and 0 <= feat_col < stride):
        raise ValueError(f"voxelize_dynamic: xyz_col={xyz_col} / feat_col={feat_col} do not fit point stride {stride}")
    f = stride - feat_col
    pc_range = np.asarray(pc_range, dtype=np.float32).reshape(-1)
    voxel_size = np.asarray(voxel_size, dtype=np.float32).reshape(-1)
    if pc_range.size != 6 or voxel_size.size != 3 or not (voxel_size > 0).all():
        raise ValueError("voxelize_dynamic: pc_range needs 6 values and voxel_size 3 positive values")
    grid = grid_size_xyz(pc_range, voxel_size) if grid is None else np.asarray(grid).reshape(-1)
    if grid.size != 3 or not (grid > 0).all():
        raise ValueError(f"voxelize_dynamic: grid must be 3 positive sizes (x, y, z), got {grid}")
    grid_c = _C.ints(grid)
    L = _C.lib()
    ws_bytes = L.toda_voxelize_dynamic_workspace_bytes(n, batch, grid_c)
    if ws_bytes == 0:
        raise RuntimeError("toda_voxelize_dynamic_workspace_bytes rejected the arguments")
    ws = _workspace("vox", ws_bytes, dev)
    features = torch.empty((max(n, 1), f), dtype=torch.float32, device=dev)
    coords = torch.empty((max(n, 1), 4), dtype=torch.int32, device=dev)
    counts = torch.empty((batch + 1,), dtype=torch.int32, device=dev)
    with _timed("voxelize_dynamic", n_points=n, batch=batch, F=f):
        rc = L.toda_voxelize_dynamic(_p(points), n, stride, xyz_col, feat_col, f, _p(frame_offsets), batch,
                                     _C.floats(pc_range), _C.floats(voxel_size), grid_c, _p(features), _p(coords),
                                     _p(counts), _p(ws), ws.numel(), _stream())
    _C.check(rc, "toda_voxelize_dynamic")
    v = int(counts[batch].item())
    return features[:v], coords[:v], counts


class _MeanVFE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, voxels, num_points):
        voxels = _need(voxels, torch.float32, "voxels")
        v, k, f = voxels.shape
        is_float = num_points.dtype == torch.float32
        if not is_float:
            num_points = _need(num_points, torch.int32, "voxel_num_points")
        num_points = num_points.contiguous()
        out = torch.empty((v, f), dtype=torch.float32, device=voxels.device)
        with _timed("mean_vfe_fwd", V=v, K=k, F=f):
            _C.check(_C.lib().toda_mean_vfe_fwd(_p(voxels), _p(num_points), int(is_float), v, k, f, _p(out), _stream()),
                     "toda_mean_vfe_fwd")
        ctx.save_for_backward(num_points)
        ctx.shape = (v, k, f, is_float)
        return out

    @staticmethod
    def backward(ctx, dout):
        (num_points,) = ctx.saved_tensors
        v, k, f, is_float = ctx.shape
        dout = dout.contiguous()
        dv = torch.empty((v, k, f), dtype=torch.float32, device=dout.device)
        _C.check(_C.lib().toda_mean_vfe_bwd(_p(dout), _p(num_points), int(is_float), v, k, f, _p(dv), _stream()),
                 "toda_mean_vfe_bwd")
        return dv, None


def mean_vfe(voxels, num_points):
    """mean_vfe.py L25-29."""
    return _MeanVFE.apply(voxels, num_points)


# ------------------------------------------------------------------------------------------------
# occupancy index + rulebooks
# ------------------------------------------------------------------------------------------------
_index_occupant = {}   # workspace key -> the OccupancyIndex whose marks are currently in that buffer


class OccupancyIndex:
    """Occupancy index over (batch, D, H, W): canonical coords + coordinate->row lookup.

    Index buffers are cached per (tag, dims) and shared: acquiring a buffer releases (un-marks) whatever
    index occupied it before, and an index that lost its buffer re-marks itself on the next use, so the
    all-zero-between-users invariant of the ABI holds without full memsets.
    """

    def __init__(self, batch, shape, device, tag):
        self.batch = int(batch)
        self.shape = [int(s) for s in shape]
        d, h, w = self.shape
        nbytes = _C.lib().toda_index_bytes(self.batch, d, h, w)
        if nbytes == 0:
            raise RuntimeError(f"bad index dims {batch} {shape}")
        self.key = (("index", tag, self.batch, d, h, w), device.index, _stream_id(device))
        self.buf = _workspace(self.key[0], nbytes, device, zero=True)
        self.coords = None
        self.frame_counts = None
        self.n = 0
        self._marked = False   # True while extra marks (not described by self.coords) may be in the buffer

    def _dims(self):
        return (self.batch, *self.shape)

    def _acquire(self):
        prev = _index_occupant.get(self.key)
        if prev is not None and prev is not self and prev.buf.data_ptr() == self.buf.data_ptr():
            prev._unmark()
        _index_occupant[self.key] = self

    def _unmark(self):
        if self.coords is not None and self.n > 0:
            _C.check(_C.lib().toda_index_release(_p(self.buf), *self._dims(), _p(self.coords), self.n, _stream()),
                     "toda_index_release")
        if _index_occupant.get(self.key) is self:
            del _index_occupant[self.key]

    def insert(self, coords):
        self._acquire()
        coords = _need(coords, torch.int32, "coords")
        _C.check(_C.lib().toda_index_insert(_p(self.buf), *self._dims(), _p(coords), coords.shape[0], _stream()),
                 "toda_index_insert")

    def insert_strided(self, in_coords, ksize, stride, padding):
        self._acquire()
        in_coords = _need(in_coords, torch.int32, "in_coords")
        _C.check(_C.lib().toda_index_insert_strided(_p(self.buf), *self._dims(), _p(in_coords), in_coords.shape[0],
                                                    _C.ints(ksize), _C.ints(stride), _C.ints(padding), _stream()),
                 "toda_index_insert_strided")

    def build(self, cap, known_n=None):
        """Ranks the marked cells; returns canonical coords (n,4).  Host sync to read n unless known_n."""
        dev = self.buf.device
        coords = torch.empty((max(cap, 1), 4), dtype=torch.int32, device=dev)
        n_out = torch.empty((self.batch + 1,), dtype=torch.int32, device=dev)
        with _timed("index_build", cells=self.batch * self.shape[0] * self.shape[1] * self.shape[2]):
            _C.check(_C.lib().toda_index_build(_p(self.buf), *self._dims(), _p(coords), cap, _p(n_out), _stream()),
                     "toda_index_build")
        self.n = int(n_out[0].item()) if known_n is None else int(known_n)
        self.coords = coords[:self.n]
        self.frame_counts = n_out
        return self.coords

    def ensure_live(self):
        """Re-marks and re-ranks this index if another index has used the shared buffer since."""
        if _index_occupant.get(self.key) is self:
            return
        if self.coords is None:
            raise RuntimeError("occupancy index was released")
        coords, n = self.coords, self.n
        self.insert(coords)
        self.build(n, known_n=n)

    def rows(self, coords):
        self.ensure_live()
        coords = _need(coords, torch.int32, "coords")
        rows = torch.empty((coords.shape[0],), dtype=torch.int32, device=coords.device)
        _C.check(_C.lib().toda_index_rows(_p(self.buf), *self._dims(), _p(coords), coords.shape[0], _p(rows), _stream()),
                 "toda_index_rows")
        return rows

    def release(self):
        if _index_occupant.get(self.key) is self:
            self._unmark()
        self.coords = None
        self.n = 0


@dataclass
class Rulebook:
    """Neighbour tables of one conv geometry (shared by every conv with the same indice_key)."""
    subm: bool
    ksize: List[int]
    stride: List[int]
    padding: List[int]
    in_shape: List[int]
    out_shape: List[int]
    n_in: int
    n_out: int
    out_coords: torch.Tensor          # (n_out,4) canonical
    nbr_fwd: torch.Tensor             # (kvol, n_out): input row per output row
    nbr_bwd: Optional[torch.Tensor]   # (kvol, n_in): output row per input row (None for SubM: mirrored nbr_fwd)
    # strided convs, for dgrad: input rows sorted by parity class (int32 (n_in,)) and nbr_bwd with its columns in that order
    dgrad_order: Optional[torch.Tensor] = None
    nbr_bwd_sorted: Optional[torch.Tensor] = None
    dgrad_tile_masks: Optional[torch.Tensor] = None   # per 128-row tile of nbr_bwd_sorted: which offsets hold a neighbour
    tile_masks: Optional[torch.Tensor] = None         # the same for nbr_fwd (forward; SubM dgrad walks the same table)
    plan: Optional["TilePlan"] = None                 # row-cache plan of nbr_fwd (forward; SubM dgrad)
    dgrad_plan: Optional["TilePlan"] = None           # row-cache plan of the strided dgrad table (nbr_bwd_sorted / nbr_bwd)

    @property
    def kvol(self):
        return self.ksize[0] * self.ksize[1] * self.ksize[2]

    def dgrad_table(self):
        """-> (nbr, out_rows, tile_masks, plan) of the dgrad: SubM walks nbr_fwd (with mirrored weights); a strided conv
        walks nbr_bwd, in parity-class order when there is one (rows written back to canonical order through out_rows)."""
        if self.subm:
            return self.nbr_fwd, None, self.tile_masks, self.plan
        if self.dgrad_order is None:
            return self.nbr_bwd, None, None, self.dgrad_plan
        return self.nbr_bwd_sorted, self.dgrad_order, self.dgrad_tile_masks, self.dgrad_plan


@dataclass
class TilePlan:
    """Row-cache plan of one neighbour table (toda_table_tile_plan): per 128-row tile and kz-group of offsets the distinct
    input rows, and the table rewritten as 16-bit slots into those lists."""
    lidx: torch.Tensor      # int16 (tiles, kvol, 128)
    rows: torch.Tensor      # int32 (tiles, ngroups, cap)
    cnt: torch.Tensor       # int32 (tiles, ngroups)
    ngroups: int
    cap: int

    def tensors(self):
        return [self.lidx, self.rows, self.cnt]


def table_tile_plan(nbr, ksize, channels):
    """Plan for the convolutions that gather `channels`-wide rows through `nbr` (None when the shape is not covered)."""
    kvol, n = nbr.shape
    ngroups = int(ksize[0])
    if n == 0 or kvol > 27 or ngroups > 3 or kvol % ngroups or kvol // ngroups > 9 or not channels:
        return None
    L = _C.lib()
    cap = L.toda_tile_plan_capacity(int(channels))
    if cap <= 0:
        return None
    tiles = (n + 127) // 128
    dev = nbr.device
    lidx = torch.empty((tiles, kvol, 128), dtype=torch.int16, device=dev)
    rows = torch.empty((tiles, ngroups, cap), dtype=torch.int32, device=dev)
    cnt = torch.empty((tiles, ngroups), dtype=torch.int32, device=dev)
    with _timed("tile_plan", n=n, kvol=kvol):
        _C.check(L.toda_table_tile_plan(_p(nbr), n, kvol, ngroups, cap, _p(lidx), _p(rows), _p(cnt), _stream()),
                 "toda_table_tile_plan")
    return TilePlan(lidx, rows, cnt, ngroups, cap)


def conv_out_size(in_size, k, s, p):
    return (in_size + 2 * p - (k - 1) - 1) // s + 1


def rulebook_subm(index: OccupancyIndex, ksize, channels=None):
    """channels: width of the rows gathered through this table (max of Cin for forward / Cout for dgrad): sizes the
    row-cache plan of the tensor-core kernel; None = no plan."""
    index.ensure_live()
    n = index.n
    kvol = ksize[0] * ksize[1] * ksize[2]
    nbr = torch.empty((kvol, n), dtype=torch.int32, device=index.buf.device)
    with _timed("rulebook_subm", n=n, kvol=kvol):
        _C.check(_C.lib().toda_rulebook_subm(_p(index.buf), index.batch, *index.shape, _p(index.coords), n, _C.ints(ksize),
                                             _p(nbr), _stream()), "toda_rulebook_subm")
    rb = Rulebook(True, list(ksize), [1, 1, 1], [k // 2 for k in ksize], index.shape, index.shape, n, n, index.coords,
                  nbr, None)
    # even in raster order a 128-row tile often has no neighbour at all under whole groups of offsets (e.g. no dz = -1 /
    # +1 neighbours on flat ground): 45 % of the K chunks at stride 1, 15-20 % deeper; the kernel skips them
    rb.tile_masks = table_tile_masks(nbr) if (n > 0 and kvol <= 32) else None
    rb.plan = table_tile_plan(nbr, ksize, channels) if _TILE_PLANS else None
    return rb


def rulebook_sparse(index_in: OccupancyIndex, ksize, stride, padding, tag, cin=None, cout=None):
    """Builds the output index (kept alive in the returned tuple) and both tables.  cin / cout size the row-cache plans
    (forward gathers Cin-wide rows through nbr_fwd, dgrad Cout-wide rows through nbr_bwd)."""
    index_in.ensure_live()
    out_shape = [conv_out_size(index_in.shape[a], ksize[a], stride[a], padding[a]) for a in range(3)]
    index_out = OccupancyIndex(index_in.batch, out_shape, index_in.buf.device, tag)
    if index_out.buf.data_ptr() == index_in.buf.data_ptr():
        # same tag and same spatial shape as the input's index (e.g. two k3 s1 p1 SparseConv3d with indice_key=None in a row):
        # acquiring the shared buffer would un-mark the input index and both tables would be built against one bitmap
        index_out = OccupancyIndex(index_in.batch, out_shape, index_in.buf.device, (tag, "alt"))
    assert index_out.buf.data_ptr() != index_in.buf.data_ptr()
    index_out.insert_strided(index_in.coords, ksize, stride, padding)
    per_in = 1
    for a in range(3):
        per_in *= min(ksize[a], (ksize[a] + stride[a] - 1) // stride[a])
    cells = index_in.batch * out_shape[0] * out_shape[1] * out_shape[2]
    cap = int(min(index_in.n * per_in, cells))
    out_coords = index_out.build(cap)
    n_in, n_out = index_in.n, index_out.n
    kvol = ksize[0] * ksize[1] * ksize[2]
    dev = index_in.buf.device
    nbr_fwd = torch.empty((kvol, n_out), dtype=torch.int32, device=dev)
    nbr_bwd = torch.empty((kvol, n_in), dtype=torch.int32, device=dev)
    with _timed("rulebook_sparse", n_in=n_in, n_out=n_out, kvol=kvol):
        _C.check(_C.lib().toda_rulebook_sparse(_p(index_in.buf), *index_in.shape, _p(index_out.buf), *out_shape,
                                               index_in.batch, _p(index_in.coords), n_in, _p(out_coords), n_out,
                                               _C.ints(ksize), _C.ints(stride), _C.ints(padding), _p(nbr_fwd), _p(nbr_bwd),
                                               _stream()), "toda_rulebook_sparse")
    rb = Rulebook(False, list(ksize), list(stride), list(padding), index_in.shape, out_shape, n_in, n_out, out_coords,
                  nbr_fwd, nbr_bwd)
    rb.tile_masks = table_tile_masks(nbr_fwd) if (n_out > 0 and kvol <= 32) else None
    rb.dgrad_order, rb.nbr_bwd_sorted = (_dgrad_parity_order(index_in.coords, nbr_bwd, stride, padding) if kvol <= 32
                                         else (None, None))
    if rb.dgrad_order is not None:
        rb.dgrad_tile_masks = table_tile_masks(rb.nbr_bwd_sorted)
    if _TILE_PLANS:
        rb.plan = table_tile_plan(nbr_fwd, ksize, cin)
        rb.dgrad_plan = table_tile_plan(rb.nbr_bwd_sorted if rb.dgrad_order is not None else nbr_bwd, ksize, cout)
    return rb, index_out


# Row-cache plans (toda_table_tile_plan) + the TMEM-operand kernel of conv_ts.cu: 14-36 % faster per layer than the round-1
# cp.async / gather4 kernels (profiles/r02_conv_ts.md), bit-identical results -- and OPT-IN (TODA_TILE_PLANS=1 or
# set_tile_plans(True)): the kernel deadlocked on some inputs (the second rank's frames, the stage-2 mixed batch) until the
# last hour of round 2, when the cause was pinned on the mbarrier.try_wait form with a suspend-time hint; with the plain form
# it has run clean since (15 bench runs), which is evidence but not a soak test (DESIGN section 6, profiles/r02_conv_ts.md
# section 5).  The default keeps the round-1 kernels, which ran every workload and 1-8 GPUs.
import os as _os
_TILE_PLANS = _os.environ.get("TODA_TILE_PLANS", "0") == "1"


def set_tile_plans(on):
    global _TILE_PLANS
    _TILE_PLANS = bool(on)


def tile_plans_enabled():
    return _TILE_PLANS


def table_tile_masks(nbr):
    """uint32 per 128-row tile of a neighbour table: bit k = some row of the tile has a neighbour under offset k."""
    kvol, n = nbr.shape
    masks = torch.empty(((n + 127) // 128,), dtype=torch.int32, device=nbr.device)
    _C.check(_C.lib().toda_table_tile_masks(_p(nbr), n, kvol, _p(masks), _stream()), "toda_table_tile_masks")
    return masks


def _dgrad_parity_order(in_coords, nbr_bwd, stride, padding):
    """Input rows of a strided conv sorted by parity class ((z+pz) % sz, (y+py) % sy, (x+px) % sx), canonical order kept
    inside a class, and the input-stationary table with its columns in that order.

    out = (in + pad - k) / stride is integral only for k = (in + pad) mod stride (+ multiples of stride), so an input voxel
    can be reached through 1..8 of the 27 offsets of a k3 s2 conv only: in canonical order every 128-row tile mixes all
    classes and the dense [27] table is ~85 % structural padding, in class order most K blocks of a tile are empty and the
    tensor-core kernel skips them (per-tile offset masks, see toda_spconv_fwd's out_rows)."""
    if all(s == 1 for s in stride) or in_coords.shape[0] == 0:
        return None, None
    if stride[0] * stride[1] * stride[2] > 8:
        return None, None
    n = in_coords.shape[0]
    L = _C.lib()
    ws = _workspace("parity", L.toda_parity_order_workspace_bytes(n), in_coords.device)
    order = torch.empty((n,), dtype=torch.int32, device=in_coords.device)
    _C.check(L.toda_parity_order(_p(in_coords), n, _C.ints(stride), _C.ints(padding), _p(order), None, _p(ws), ws.numel(),
                                 _stream()), "toda_parity_order")
    return order, nbr_bwd.index_select(1, order).contiguous()


# ------------------------------------------------------------------------------------------------
# K5-K7 sparse convolution
# ------------------------------------------------------------------------------------------------
_repack_cache = {}


def invalidate_weight_cache():
    """Drops the cached weight repacks.  The cache is validated by the parameter's autograd version counter, which
    in-place writes through `.data` (pcdet's OptimWrapper true-weight-decay path `p.data.mul_()`, EMA / SWA swaps,
    `.data.copy_()`) do NOT bump: call this after such an update (or after loading a checkpoint into live modules)."""
    _repack_cache.clear()


def _repack(weight, transpose, mirror, want_bf16=False):
    """[kvol][Cin][Cout] (or transposed / k-mirrored) copy of a (Cout,kz,ky,kx,Cin) parameter, cached until the
    parameter is modified (optimizer step bumps ._version; for `.data` writes see invalidate_weight_cache).
    want_bf16: -> (fp32 repack, K-major bf16 copy for the tensor-core kernels (toda_weight_kmajor_bf16), cached alongside)."""
    key = (id(weight), bool(transpose), bool(mirror))
    hit = _repack_cache.get(key)
    if hit is not None and hit[2]() is weight and hit[0] == weight._version and hit[3] == weight.data_ptr():
        out = hit[1]
    else:
        cout, kvol, cin = weight.shape[0], weight.shape[1] * weight.shape[2] * weight.shape[3], weight.shape[4]
        out = torch.empty((kvol, cout, cin) if transpose else (kvol, cin, cout), dtype=torch.float32, device=weight.device)
        _C.check(_C.lib().toda_weight_repack(_p(weight), kvol, cin, cout, int(transpose), int(mirror), _p(out), _stream()),
                 "toda_weight_repack")
        if len(_repack_cache) > 512:
            _repack_cache.clear()
        hit = [weight._version, out, weakref.ref(weight), weight.data_ptr(), None]
        _repack_cache[key] = hit
    if not want_bf16:
        return out
    if hit[4] is None:
        kvol, ci, co = out.shape
        wb = torch.empty((co, kvol * max(ci, 16)), dtype=torch.bfloat16, device=out.device)
        _C.check(_C.lib().toda_weight_kmajor_bf16(_p(out), kvol, ci, co, _p(wb), _stream()), "toda_weight_kmajor_bf16")
        hit[4] = wb
    return out, hit[4]


def _bf16_shadow_of(t):
    """bf16 copy attached to a gradient tensor by the BN backward pass (valid only if the tensor was not modified since)."""
    tag = getattr(t, "_toda_bf16", None)
    if tag is not None and tag[1] == t._version and tag[0].shape == t.shape:
        return tag[0]
    return None


def _conv_call(x, xb, cin, nbr, n_out, kvol, w, cout, bias, precision, what="conv_fwd", rb=None, bn_sums=None, y=None,
               out_rows=None, tile_masks=None, plan=None, addend=None, w_bf16=None):
    """addend (optional, (n_out, cout) fp32): added to the result in the kernel's epilogue."""
    if y is None:
        y = torch.empty((n_out, cout), dtype=torch.float32, device=x.device)
    L = _C.lib()
    ws_bytes = L.toda_spconv_fwd_workspace_bytes(x.shape[0], cin, cout, kvol, precision)
    ws = _workspace("conv", ws_bytes, x.device) if ws_bytes else None
    with _timed(what, n_in=x.shape[0], n_out=n_out, cin=cin, cout=cout, kvol=kvol, precision=precision, rb=id(rb)):
        _C.check(L.toda_spconv_fwd(_p(x), _p(xb), x.shape[0], cin, _p(nbr), n_out, kvol, _p(w), cout, _p(bias), _p(addend), _p(y),
                                   _p(out_rows), _p(tile_masks), _p(plan.lidx) if plan else None,
                                   _p(plan.rows) if plan else None, _p(plan.cnt) if plan else None,
                                   plan.ngroups if plan else 0, plan.cap if plan else 0, _p(bn_sums), _p(w_bf16), precision,
                                   _p(ws), ws.numel() if ws is not None else 0, _stream()), "toda_spconv_fwd")
    return y


def _conv_forward_impl(x, x_bf16, weight, bias, rb, precision, want_stats):
    """-> (y, sums, x, weight, x_bf16): the conv output, the fused BN sums (or None) and the tensors backward needs."""
    x = _need(x.contiguous(), torch.float32, "features")
    weight = _need(weight.contiguous(), torch.float32, "weight")
    cout, cin = weight.shape[0], weight.shape[4]
    assert x.shape == (rb.n_in, cin), (x.shape, rb.n_in, cin)
    if x_bf16 is not None and (precision != CONV_BF16 or x_bf16.shape != x.shape or x_bf16.dtype != torch.bfloat16
                               or not x_bf16.is_contiguous()):
        x_bf16 = None
    w = _repack(weight, False, False)
    b = bias.contiguous() if bias is not None else None
    sums = None
    if want_stats and rb.n_out > 0 and _C.lib().toda_spconv_uses_tensor_cores(cin, cout, rb.kvol, precision):
        sums = torch.empty((2 * cout,), dtype=torch.float64, device=x.device)
    y = _conv_call(x, x_bf16, cin, rb.nbr_fwd, rb.n_out, rb.kvol, w, cout, b, precision, "conv_fwd", rb, sums,
                   tile_masks=rb.tile_masks, plan=rb.plan)
    return y, sums, x, weight, x_bf16


def _conv_backward_impl(dy, dyb, x, weight, xb, rb, precision, need_dx, need_dw, need_db):
    cout, cin = weight.shape[0], weight.shape[4]
    L = _C.lib()
    dx = dw = db = None
    if need_dx:
        # dgrad = the same gather-GEMM on the input-stationary table with transposed weights
        wt = _repack(weight, True, rb.subm)
        nbr, out_rows, masks, plan = rb.dgrad_table()
        dx = _conv_call(dy, dyb, cout, nbr, rb.n_in, rb.kvol, wt, cin, None, precision, "conv_dgrad", rb,
                        out_rows=out_rows, tile_masks=masks, plan=plan)
    if need_dw:
        dw = torch.empty_like(weight)
        ws_bytes = L.toda_spconv_wgrad_workspace_bytes(rb.n_in, rb.n_out, rb.kvol, cin, cout, precision)
        ws = _workspace("wgrad", ws_bytes, dy.device)
        with _timed("conv_wgrad", n_in=rb.n_in, n_out=rb.n_out, cin=cin, cout=cout, kvol=rb.kvol, precision=precision,
                    rb=id(rb)):
            _C.check(L.toda_spconv_wgrad(_p(x), _p(xb), rb.n_in, cin, _p(rb.nbr_fwd), rb.n_out, rb.kvol, _p(rb.tile_masks),
                                         _p(dy), _p(dyb), cout, _p(dw), _p(ws), ws.numel(), precision, _stream()),
                     "toda_spconv_wgrad")
    if need_db:
        db = col_sum(dy)
    return dx, dw, db


class _SparseConv(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, x_bf16, weight, bias, rb: Rulebook, precision, want_stats):
        y, sums, x, weight, x_bf16 = _conv_forward_impl(x, x_bf16, weight, bias, rb, precision, want_stats)
        ctx.save_for_backward(x, weight, x_bf16)
        ctx.set_materialize_grads(False)      # no zero tensors for the non-differentiable outputs
        ctx.rb, ctx.precision, ctx.has_bias = rb, precision, bias is not None
        if sums is not None:
            ctx.mark_non_differentiable(sums)
        return y, sums

    @staticmethod
    def backward(ctx, dy, _dsums=None):
        if dy is None:
            return (None,) * 7
        x, weight, xb = ctx.saved_tensors
        dyb = _bf16_shadow_of(dy) if (ctx.precision == CONV_BF16 and dy.is_contiguous()) else None
        dx, dw, db = _conv_backward_impl(dy.contiguous(), dyb, x, weight, xb, ctx.rb, ctx.precision, ctx.needs_input_grad[0],
                                         ctx.needs_input_grad[2], ctx.has_bias and ctx.needs_input_grad[3])
        return dx, None, dw, db, None, None, None


def sparse_conv(x, weight, bias, rb, precision=CONV_FP32, x_bf16=None, want_stats=False):
    """y = conv(x).  want_stats: also return the per-channel (sum, sum of squares) of y accumulated by the kernel's
    epilogue (double[2*Cout], or None when this shape does not run on the tensor-core kernel) for bn_act(sums=...)."""
    y, sums = _SparseConv.apply(x, x_bf16, weight, bias, rb, precision, want_stats)
    return (y, sums) if want_stats else y


def col_sum(t):
    n, c = t.shape
    out = torch.empty((c,), dtype=torch.float32, device=t.device)
    L = _C.lib()
    ws = _workspace("bn", L.toda_bn_workspace_bytes(c), t.device)
    _C.check(L.toda_col_sum(_p(t), n, c, _p(out), _p(ws), ws.numel(), _stream()), "toda_col_sum")
    return out


# ------------------------------------------------------------------------------------------------
# K8 BatchNorm + ReLU (+ residual)
# ------------------------------------------------------------------------------------------------
class ReluMaskTape:
    """Test instrument (tests/test_gpu_tc.py): records the ReLU masks of one pass ('record') and imposes them on another
    ('replay'), so that two arithmetic modes can be compared with identical activation patterns -- the mask flips of a
    perturbed forward pass otherwise dominate any end-to-end gradient comparison.  Not used on the product path."""

    def __init__(self, mode):
        assert mode in ("record", "replay")
        self.mode, self.masks, self.i = mode, [], 0

    def replay(self):
        self.mode, self.i = "replay", 0
        return self


_relu_tape = None


def set_relu_mask_tape(tape):
    global _relu_tape
    _relu_tape = tape


# ------------------------------------------------------------------------------------------------
# BatchNorm synchronized across processes (torch.nn.SyncBatchNorm)
# ------------------------------------------------------------------------------------------------
def sync_group(bn):
    """The process group over which `bn` reduces its batch statistics in this call, or None for a local BatchNorm.
    torch.nn.SyncBatchNorm's rule (torch 2.11): a SyncBatchNorm in training mode synchronizes when torch.distributed is
    initialized and its process_group (None: WORLD) has more than one rank; otherwise it is an ordinary BatchNorm1d."""
    if not isinstance(bn, torch.nn.SyncBatchNorm) or not bn.training:
        return None
    if bn.momentum is None:
        raise NotImplementedError("toda_b200: SyncBatchNorm with momentum=None (cumulative moving average) is not supported; "
                                  "set a momentum (these backbones use 0.01)")
    if not (dist.is_available() and dist.is_initialized()):
        return None
    group = bn.process_group if bn.process_group is not None else dist.group.WORLD
    return group if dist.get_world_size(group) > 1 else None


def _run_phases(phases, group):
    """Drives a phase generator (_bn_forward_phases, _bn_backward_phases, _layer_forward_phases, _layer_backward_phases):
    every buffer it yields -- only a synchronized BatchNorm's do -- is all-reduced (SUM over `group`, in place, on the current stream: NCCL orders it after
    the local kernels without a host synchronisation) before the generator continues.  Returns the generator's result."""
    try:
        buf = next(phases)
        while True:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
            buf = phases.send(None)
    except StopIteration as stop:
        return stop.value


def _tape_mask(a, want_bf16):
    """The ReluMaskTape's mask on a pre-activation `a` -> (a, a_bf16, mask as float32)."""
    if _relu_tape.mode == "record":
        mask = a > 0
        _relu_tape.masks.append(mask)
    else:
        mask = _relu_tape.masks[_relu_tape.i]
        _relu_tape.i += 1
    a = a * mask
    return a, (a.to(torch.bfloat16) if want_bf16 else None), mask.to(torch.float32)


def _bn_forward_phases(y, gamma, beta, running_mean, running_var, eps, momentum, training, residual, relu, want_bf16, sums,
                       need_grad, sync=False):
    """Phase generator (see _run_phases) of BatchNorm (+ residual) (+ ReLU) over y.  Training: the fp64 sums of y (the conv
    epilogue's `sums` when given), yielded with the row count for the all-reduce when `sync`, then one apply that derives
    the coefficients and running statistics from them.  -> (a, a_bf16, y, mean, rstd, a_mask, global_sums): a_mask is what
    the backward pass derives the ReLU mask from (`a` itself, except under a ReluMaskTape); global_sums is the all-reduced
    buffer (None unless sync)."""
    y = _need(y.contiguous(), torch.float32, "bn input")
    n, c = y.shape
    dev = y.device
    L = _C.lib()
    scale, shift, mean, rstd = torch.empty((4, c), dtype=torch.float32, device=dev).unbind(0)
    gsums = count = None
    if training:
        if sync or sums is None:
            buf = torch.empty((2 * c + 1 if sync else 2 * c,), dtype=torch.float64, device=dev)
            count = buf.data_ptr() + 16 * c if sync else None
            ws = _workspace("bn", L.toda_bn_workspace_bytes(c), dev)
            with _timed("bn_stats", n=n, c=c):
                _C.check(L.toda_bn_local_sums(_p(y), _p(sums), n, c, _p(buf), count, _p(ws), ws.numel(), _stream()),
                         "toda_bn_local_sums")
            sums = buf
        if sync:
            yield sums
            gsums = sums
    else:
        _C.check(L.toda_bn_eval_coeffs(_p(gamma), _p(beta), _p(running_mean), _p(running_var), float(eps), c, _p(scale),
                                       _p(shift), _stream()), "toda_bn_eval_coeffs")
        mean = running_mean
        rstd = torch.rsqrt(running_var + eps) if need_grad else None
    res = residual.contiguous() if residual is not None else None
    a = torch.empty_like(y)
    tape = _relu_tape is not None and relu      # pre-activation z, then the recorded / replayed mask (see ReluMaskTape)
    ab = torch.empty(y.shape, dtype=torch.bfloat16, device=dev) if (want_bf16 and not tape) else None
    act = 0 if tape else int(relu)
    with _timed("bn_apply", n=n, c=c, residual=res is not None):
        if training:
            _C.check(L.toda_bn_apply_sums(_p(y), n, c, _p(sums), count, _p(gamma), _p(beta), float(eps), float(momentum),
                                          _p(running_mean), _p(running_var), _p(scale), _p(shift), _p(mean), _p(rstd), _p(res),
                                          act, _p(a), _p(ab), _stream()), "toda_bn_apply_sums")
        else:
            _C.check(L.toda_bn_apply(_p(y), n, c, _p(scale), _p(shift), _p(res), act, _p(a), _p(ab), _stream()), "toda_bn_apply")
    if tape:
        a, ab, mask = _tape_mask(a, want_bf16)
        return a, ab, y, mean, rstd, mask, gsums
    return a, ab, y, mean, rstd, a, gsums


def _bn_backward_phases(da, y, a, gamma, mean, rstd, training, relu, has_res, want_bf16, gsums=None, want_db=False):
    """Phase generator of the backward of _bn_forward_phases -> (dy, dy_bf16, dresidual, dgamma, dbeta, dbias).  gsums: the
    forward's global sums of a synchronized BatchNorm: the local sums of g and g*xhat (and this process's dgamma / dbeta) are
    then yielded for the all-reduce, and dy follows from the global sums and the forward's global count.  da None = zeros (a
    rank must join the collective even when no gradient reached it).  want_db: dbias = the column sums of dy (the gradient
    of the preceding convolution's bias), summed by the pass that writes dy; else None."""
    n, c = y.shape
    da = da.contiguous() if da is not None else torch.zeros_like(y)
    L = _C.lib()
    dy = torch.empty_like(y)
    dyb = torch.empty(y.shape, dtype=torch.bfloat16, device=y.device) if want_bf16 else None
    dres = torch.empty_like(y) if has_res else None
    dgamma, dbeta = torch.empty((2, c), dtype=torch.float32, device=y.device).unbind(0)
    db = torch.empty((c,), dtype=torch.float32, device=y.device) if want_db else None
    ws = _workspace("bn", L.toda_bn_workspace_bytes(c), y.device)
    if gsums is None:
        with _timed("bn_bwd", n=n, c=c, residual=has_res):
            _C.check(L.toda_bn_bwd(_p(da), _p(a), _p(y), n, c, _p(gamma), _p(mean), _p(rstd), int(relu), int(training),
                                   _p(dy), _p(dyb), _p(dres), _p(dgamma), _p(dbeta), _p(db), _p(ws), ws.numel(), _stream()),
                     "toda_bn_bwd")
        return dy, dyb, dres, dgamma, dbeta, db
    red = torch.empty((2 * c,), dtype=torch.float64, device=y.device)
    _C.check(L.toda_bn_bwd_reduce(_p(da), _p(a), _p(y), n, c, _p(mean), _p(rstd), int(relu), _p(red), _p(dgamma), _p(dbeta),
                                  _p(ws), ws.numel(), _stream()), "toda_bn_bwd_reduce")
    yield red
    _C.check(L.toda_bn_bwd_finish(_p(da), _p(a), _p(y), n, c, _p(gamma), _p(mean), _p(rstd), int(relu), 1, _p(red),
                                  gsums.data_ptr() + 16 * c, _p(dy), _p(dyb), _p(dres), _p(db), _p(ws), ws.numel(), _stream()),
             "toda_bn_bwd_finish")
    return dy, dyb, dres, dgamma, dbeta, db


class _BNAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, gamma, beta, running_mean, running_var, eps, momentum, training, residual, relu, want_bf16, sums, group):
        a, ab, y, mean, rstd, a_mask, gsums = _run_phases(
            _bn_forward_phases(y, gamma, beta, running_mean, running_var, eps, momentum, training, residual, relu, want_bf16, sums,
                        y.requires_grad or gamma.requires_grad, group is not None), group)
        ctx.save_for_backward(y, a_mask, gamma, mean, rstd, gsums)
        ctx.set_materialize_grads(False)      # the bf16 copy is non-differentiable: no zero tensor for it in backward
        ctx.cfg = (bool(training), bool(relu), residual is not None, bool(want_bf16))
        ctx.group = group
        if ab is not None:
            ctx.mark_non_differentiable(ab)
        return a, ab

    @staticmethod
    def backward(ctx, da, _dab=None):
        if da is None and ctx.group is None:      # a synchronized BatchNorm still joins its peers' collective
            return (None,) * 13
        y, a, gamma, mean, rstd, gsums = ctx.saved_tensors
        training, relu, has_res, want_bf16 = ctx.cfg
        dy, dyb, dres, dgamma, dbeta, _ = _run_phases(_bn_backward_phases(da, y, a, gamma, mean, rstd, training, relu, has_res,
                                                                          want_bf16, gsums), ctx.group)
        if dyb is not None:
            dy._toda_bf16 = (dyb, dy._version)     # picked up by the producing conv's backward (see _bf16_shadow_of)
        return dy, dgamma, dbeta, None, None, None, None, None, dres, None, None, None, None


def _vp(t):
    return t.data_ptr() if t is not None else None


def _fused_ok(training, need_grad):
    """The one-call-per-layer C path (toda_layer_fwd / toda_layer_bwd) is used unless a per-kernel profile pass or the
    ReLU-mask test instrument is active, or a gradient is wanted through eval-mode BatchNorm (kept on the stepwise path)."""
    return _prof is None and _relu_tape is None and (training or not need_grad)


def _layer_forward(x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps, momentum, training,
                   residual, relu, want_bf16, need_grad=True, group=None):
    """conv -> BN (+residual) (+ReLU).  -> (a, a_bf16, saved) with saved = (x, x_bf16, weight, y, a_mask, gamma, mean, rstd,
    global_sums).  group: the process group of a synchronized BatchNorm (sync_group), else None (global_sums is then None)."""
    return _run_phases(_layer_forward_phases(x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps,
                                             momentum, residual, relu, want_bf16, need_grad, training, group is not None), group)


def _layer_forward_phases(x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps, momentum,
                          residual, relu, want_bf16, need_grad=True, training=True, sync=True):
    """Phase generator (see _run_phases) of _layer_forward.  sync: the BatchNorm is synchronized across processes; the local
    sums (double[2C+1], with the row count) are then yielded for the all-reduce between toda_layer_fwd_stats and
    toda_layer_fwd_apply (else one toda_layer_fwd call, and global_sums is None)."""
    if not _fused_ok(training, need_grad):
        y, sums, x, weight, x_bf16 = _conv_forward_impl(x, x_bf16, weight, bias, rb, precision, bool(training))
        a, ab, y, mean, rstd, a_mask, gsums = yield from _bn_forward_phases(y, gamma, beta, running_mean, running_var, eps,
                                                                            momentum, training, residual, relu, want_bf16, sums,
                                                                            need_grad, sync)
        return a, ab, (x, x_bf16, weight, y, a_mask, gamma, mean, rstd, gsums)
    args, x, x_bf16, weight, y, a, ab, small, _keep = _layer_fwd_args(
        x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps, momentum, training, residual, relu,
        want_bf16)
    cout = y.shape[1]
    L = _C.lib()
    gsums = None
    if sync:
        gsums = torch.empty((2 * cout + 1,), dtype=torch.float64, device=y.device)
        _C.check(L.toda_layer_fwd_stats(ctypes.byref(args), _p(gsums), _stream()), "toda_layer_fwd_stats")
        yield gsums
        _C.check(L.toda_layer_fwd_apply(ctypes.byref(args), _p(gsums), _stream()), "toda_layer_fwd_apply")
    else:
        _C.check(L.toda_layer_fwd(ctypes.byref(args), _stream()), "toda_layer_fwd")
    mean = small[2 * cout:3 * cout] if training else running_mean
    rstd = small[3 * cout:4 * cout] if training else None
    return a, ab, (x, x_bf16, weight, y, a, gamma, mean, rstd, gsums)


def _layer_fwd_args(x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps, momentum, training,
                    residual, relu, want_bf16):
    """Outputs and toda_layer_fwd_args of one fused layer -> (args, x, x_bf16, weight, y, a, a_bf16, small, keep); keep
    holds the other tensors the args point to: all of them must stay alive until the layer's calls are enqueued."""
    x = _need(x.contiguous(), torch.float32, "features")
    weight = _need(weight.contiguous(), torch.float32, "weight")
    cout, cin = weight.shape[0], weight.shape[4]
    assert x.shape == (rb.n_in, cin), (x.shape, rb.n_in, cin)
    if x_bf16 is not None and (precision != CONV_BF16 or x_bf16.shape != x.shape or x_bf16.dtype != torch.bfloat16
                               or not x_bf16.is_contiguous()):
        x_bf16 = None
    L = _C.lib()
    kvol, n_out, dev = rb.kvol, rb.n_out, x.device
    tc = bool(L.toda_spconv_uses_tensor_cores(cin, cout, kvol, precision))
    if tc and precision == CONV_BF16:
        w, wb = _repack(weight, False, False, True)
    else:
        w, wb = _repack(weight, False, False), None
    y = torch.empty((n_out, cout), dtype=torch.float32, device=dev)
    a = torch.empty_like(y)
    ab = torch.empty((n_out, cout), dtype=torch.bfloat16, device=dev) if want_bf16 else None
    small = torch.empty((8 * cout,), dtype=torch.float32, device=dev)       # scale, shift, mean, rstd | sums (2c doubles)
    ws_bytes = L.toda_spconv_fwd_workspace_bytes(x.shape[0], cin, cout, kvol, precision)
    ws = _workspace("conv", ws_bytes, dev) if ws_bytes else None
    bws = _workspace("bn", L.toda_bn_workspace_bytes(cout), dev)
    res = residual.contiguous() if residual is not None else None
    b = bias.contiguous() if bias is not None else None
    pl = rb.plan
    sp = small.data_ptr()
    args = _C.LayerFwdArgs(
        x.data_ptr(), _vp(x_bf16), x.shape[0], cin, rb.nbr_fwd.data_ptr(), n_out, kvol, w.data_ptr(), _vp(wb), cout, _vp(b),
        _vp(rb.tile_masks), _vp(pl.lidx) if pl else None, _vp(pl.rows) if pl else None, _vp(pl.cnt) if pl else None,
        pl.ngroups if pl else 0, pl.cap if pl else 0, precision, _vp(ws), ws.numel() if ws is not None else 0,
        gamma.data_ptr(), beta.data_ptr(), float(eps), float(momentum), _vp(running_mean), _vp(running_var), int(bool(training)),
        _vp(res), int(bool(relu)), y.data_ptr(), sp + 16 * cout, sp, a.data_ptr(), _vp(ab), bws.data_ptr(), bws.numel())
    return args, x, x_bf16, weight, y, a, ab, small, (w, wb, ws, bws, res, b)


def _layer_backward(da, saved, rb, precision, training, relu, has_res, has_bias, need_dx, need_dw, addend=None, group=None):
    """-> (dx, dw, db, dgamma, dbeta, dres).  addend: a gradient to be ADDED to dx (fused into the dgrad epilogue).
    group: the process group of a synchronized BatchNorm (then da may be None: zeros)."""
    return _run_phases(_layer_backward_phases(da, saved, rb, precision, relu, has_res, has_bias, need_dx, need_dw, addend,
                                              training), group)


def _layer_backward_phases(da, saved, rb, precision, relu, has_res, has_bias, need_dx, need_dw, addend=None, training=True):
    """Phase generator of _layer_backward.  With a synchronized BatchNorm (global_sums in `saved`) the local sums of g and
    g*xhat (double[2C]) are yielded for the all-reduce between toda_layer_bwd_reduce and toda_layer_bwd_finish, and dy uses
    the forward's global count; dgamma / dbeta are this process's own (as torch.nn.SyncBatchNorm's: the gradient all-reduce
    averages them)."""
    x, xb, weight, y, a_mask, gamma, mean, rstd, gsums = saved
    if da is None:
        da = torch.zeros_like(y)
    if not _fused_ok(training, True):
        dy, dyb, dres, dgamma, dbeta, db = yield from _bn_backward_phases(da, y, a_mask, gamma, mean, rstd, training, relu,
                                                                          has_res, precision == CONV_BF16, gsums, has_bias)
        dx, dw, _ = _conv_backward_impl(dy, dyb, x, weight, xb, rb, precision, need_dx, need_dw, False)
        if addend is not None and dx is not None:
            dx = dx + addend
        return dx, dw, db, dgamma, dbeta, dres
    args, dx, dw, dres, small, _keep = _layer_bwd_args(da, saved, rb, precision, training, relu, has_res, has_bias, need_dx,
                                                       need_dw, addend)
    cout = y.shape[1]
    L = _C.lib()
    if gsums is None:
        _C.check(L.toda_layer_bwd(ctypes.byref(args), _stream()), "toda_layer_bwd")
    else:
        red = torch.empty((2 * cout,), dtype=torch.float64, device=y.device)
        _C.check(L.toda_layer_bwd_reduce(ctypes.byref(args), _p(red), _stream()), "toda_layer_bwd_reduce")
        yield red
        _C.check(L.toda_layer_bwd_finish(ctypes.byref(args), _p(red), gsums.data_ptr() + 16 * cout, _stream()),
                 "toda_layer_bwd_finish")
    return dx, dw, (small[2 * cout:] if has_bias else None), small[:cout], small[cout:2 * cout], dres


def _layer_bwd_args(da, saved, rb, precision, training, relu, has_res, has_bias, need_dx, need_dw, addend):
    """Outputs and toda_layer_bwd_args of one fused layer's backward -> (args, dx, dw, dres, small, keep): small = dgamma,
    dbeta, dbias; keep holds the other tensors the args point to."""
    x, xb, weight, y, a_mask, gamma, mean, rstd, _ = saved
    L = _C.lib()
    da = da.contiguous()
    n_out, cout = y.shape
    cin, kvol, dev = weight.shape[4], rb.kvol, y.device
    bf16 = precision == CONV_BF16
    dy = torch.empty_like(y)
    dyb = torch.empty(y.shape, dtype=torch.bfloat16, device=dev) if bf16 else None
    dres = torch.empty_like(y) if has_res else None
    small = torch.empty((3 * cout,), dtype=torch.float32, device=dev)        # dgamma, dbeta, dbias
    bws = _workspace("bn", L.toda_bn_workspace_bytes(cout), dev)
    dx = dw = None
    wt = wtb = None
    nbr = out_rows = masks = pl = None
    if need_dx:
        tc = bool(L.toda_spconv_uses_tensor_cores(cout, cin, kvol, precision))
        if tc and precision == CONV_BF16:
            wt, wtb = _repack(weight, True, rb.subm, True)
        else:
            wt = _repack(weight, True, rb.subm)
        nbr, out_rows, masks, pl = rb.dgrad_table()
        dx = torch.empty((rb.n_in, cin), dtype=torch.float32, device=dev)
        if addend is not None:
            addend = addend.contiguous()
    ws_bytes = L.toda_spconv_fwd_workspace_bytes(n_out, cout, cin, kvol, precision) if need_dx else 0
    ws = _workspace("conv", ws_bytes, dev) if ws_bytes else None
    wws = None
    if need_dw:
        dw = torch.empty_like(weight)
        wws = _workspace("wgrad", L.toda_spconv_wgrad_workspace_bytes(rb.n_in, n_out, kvol, cin, cout, precision), dev)
    sp = small.data_ptr()
    args = _C.LayerBwdArgs(
        da.data_ptr(), a_mask.data_ptr(), y.data_ptr(), n_out, cout, gamma.data_ptr(), _vp(mean), _vp(rstd), int(relu), int(training),
        dy.data_ptr(), _vp(dyb), _vp(dres), sp, sp + 4 * cout, bws.data_ptr(), bws.numel(),
        x.data_ptr(), _vp(xb), rb.n_in, cin, kvol,
        int(bool(need_dx)), _vp(nbr), _vp(wt), _vp(wtb), _vp(out_rows), _vp(masks),
        _vp(pl.lidx) if pl else None, _vp(pl.rows) if pl else None, _vp(pl.cnt) if pl else None, pl.ngroups if pl else 0,
        pl.cap if pl else 0, _vp(addend) if need_dx else None, _vp(dx),
        int(bool(need_dw)), rb.nbr_fwd.data_ptr(), _vp(rb.tile_masks), _vp(dw), _vp(wws), wws.numel() if wws is not None else 0,
        int(bool(has_bias)), sp + 8 * cout, precision, _vp(ws), ws.numel() if ws is not None else 0)
    return args, dx, dw, dres, small, (da, dy, dyb, addend, wt, wtb, ws, wws, bws)


class _ConvBNAct(torch.autograd.Function):
    """conv -> BatchNorm1d (+ residual) (+ ReLU) as ONE autograd node and ONE C call each way (toda_layer_fwd / _bwd): the
    gradient between BN and conv (dy and its bf16 copy) never becomes a graph edge."""

    @staticmethod
    def forward(ctx, x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps, momentum, training,
                residual, relu, want_bf16, group):
        need_grad = any(ctx.needs_input_grad)
        a, ab, saved = _layer_forward(x, x_bf16, weight, bias, rb, precision, gamma, beta, running_mean, running_var, eps, momentum,
                                      training, residual, relu, want_bf16, need_grad, group)
        if need_grad:
            ctx.save_for_backward(*saved)
        ctx.set_materialize_grads(False)
        ctx.rb, ctx.precision, ctx.has_bias, ctx.group = rb, precision, bias is not None, group
        ctx.cfg = (bool(training), bool(relu), residual is not None, bool(want_bf16))
        if ab is not None:
            ctx.mark_non_differentiable(ab)
        return a, ab

    @staticmethod
    def backward(ctx, da, _dab=None):
        if da is None and ctx.group is None:      # a synchronized BatchNorm still joins its peers' collective
            return (None,) * 17
        training, relu, has_res, want_bf16 = ctx.cfg
        dx, dw, db, dgamma, dbeta, dres = _layer_backward(da, ctx.saved_tensors, ctx.rb, ctx.precision, training, relu, has_res,
                                                          ctx.has_bias and ctx.needs_input_grad[3], ctx.needs_input_grad[0],
                                                          ctx.needs_input_grad[2], group=ctx.group)
        return dx, None, dw, db, None, None, dgamma, dbeta, None, None, None, None, None, dres, None, None, None


class _ResBlock(torch.autograd.Function):
    """SparseBasicBlock (spconv_backbone.py L30-66) as one autograd node: conv1-bn1-relu, conv2-bn2, + identity, relu.
    Backward: layer 2, then layer 1 with the residual-branch gradient added in its dgrad epilogue (no separate add pass,
    no autograd accumulation of the two branches)."""

    @staticmethod
    def forward(ctx, x, x_bf16, w1, b1, g1, be1, rm1, rv1, w2, b2, g2, be2, rm2, rv2, rb, precision, eps, momentum, training, want_bf16,
                group1, group2):
        need_grad = any(ctx.needs_input_grad)
        h, hb, s1 = _layer_forward(x, x_bf16, w1, b1, rb, precision, g1, be1, rm1, rv1, eps, momentum, training, None, True,
                                   want_bf16, need_grad, group1)
        out, outb, s2 = _layer_forward(h, hb, w2, b2, rb, precision, g2, be2, rm2, rv2, eps, momentum, training, s1[0], True,
                                       want_bf16, need_grad, group2)
        if need_grad:
            ctx.save_for_backward(*s1, *s2)
        ctx.set_materialize_grads(False)
        ctx.rb, ctx.precision, ctx.training = rb, precision, bool(training)
        ctx.groups = (group1, group2)
        ctx.has_bias = (b1 is not None, b2 is not None)
        if outb is not None:
            ctx.mark_non_differentiable(outb)
        return out, outb

    @staticmethod
    def backward(ctx, dout, _db=None):
        if dout is None and ctx.groups == (None, None):      # a synchronized BatchNorm still joins its peers' collectives
            return (None,) * 22
        sv = ctx.saved_tensors
        s1, s2 = sv[:9], sv[9:]
        ng = ctx.needs_input_grad
        dh, dw2, db2, dg2, dbe2, dres = _layer_backward(dout, s2, ctx.rb, ctx.precision, ctx.training, True, True,
                                                        ctx.has_bias[1] and ng[9], True, ng[8], group=ctx.groups[1])
        dx, dw1, db1, dg1, dbe1, _ = _layer_backward(dh, s1, ctx.rb, ctx.precision, ctx.training, True, False,
                                                     ctx.has_bias[0] and ng[3], ng[0], ng[2], addend=dres if ng[0] else None,
                                                     group=ctx.groups[0])
        return (dx, None, dw1, db1, dg1, dbe1, None, None, dw2, db2, dg2, dbe2, None, None, None, None, None, None, None, None,
                None, None)


def _bn_call(bn):
    """-> (training, group) of one call of BatchNorm module `bn` (group: see sync_group); a training call counts the batch
    in num_batches_tracked, as torch.nn.BatchNorm1d does."""
    group = sync_group(bn)
    training = bn.training or bn.running_mean is None
    if training and bn.running_mean is not None and bn.num_batches_tracked is not None:
        bn.num_batches_tracked += 1
    return training, group


def res_block(x, x_bf16, conv1_w, conv1_b, bn1, conv2_w, conv2_b, bn2, rb, precision, want_bf16=False):
    """SparseBasicBlock on feature rows; bn1 / bn2 are the nn.BatchNorm1d (or nn.SyncBatchNorm) modules.
    -> (out, out_bf16 or None)"""
    (training, group1), (training2, group2) = _bn_call(bn1), _bn_call(bn2)
    assert bn1.eps == bn2.eps and bn1.momentum == bn2.momentum and training == training2
    return _ResBlock.apply(x, x_bf16, conv1_w, conv1_b, bn1.weight, bn1.bias, bn1.running_mean, bn1.running_var, conv2_w, conv2_b,
                           bn2.weight, bn2.bias, bn2.running_mean, bn2.running_var, rb, precision, bn1.eps, bn1.momentum, training,
                           want_bf16, group1, group2)


def conv_bn_act(x, weight, bias, rb, precision, bn: torch.nn.BatchNorm1d, residual=None, relu=True, x_bf16=None, want_bf16=False):
    """Fused-node version of bn_act(sparse_conv(x, ...), bn, residual, relu).  -> (a, a_bf16 or None).  An nn.SyncBatchNorm
    in training mode reduces its statistics over its process group (sync_group)."""
    training, group = _bn_call(bn)
    return _ConvBNAct.apply(x, x_bf16, weight, bias, rb, precision, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps,
                            bn.momentum, training, residual, relu, want_bf16, group)


def bn_act(y, bn: torch.nn.BatchNorm1d, residual=None, relu=True, want_bf16=False, sums=None):
    """BatchNorm1d (+ residual) (+ ReLU) with the module's parameters / running stats
    (spconv_backbone.py L23-24, L54-64).  want_bf16: also return the bf16 copy written by the same pass.
    sums: per-channel (sum, sum of squares) of y from the producing convolution's epilogue (skips the statistics pass).
    An nn.SyncBatchNorm in training mode reduces its statistics over its process group (sync_group)."""
    training, group = _bn_call(bn)
    a, ab = _BNAct.apply(y, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, bn.momentum, training, residual,
                         relu, want_bf16, sums if training else None, group)
    return (a, ab) if want_bf16 else a


# ------------------------------------------------------------------------------------------------
# K9 BEV scatter
# ------------------------------------------------------------------------------------------------
class _BEVScatter(torch.autograd.Function):
    @staticmethod
    def forward(ctx, features, coords, batch, d, h, w):
        features = _need(features.contiguous(), torch.float32, "features")
        coords = _need(coords, torch.int32, "indices")
        n, c = features.shape
        out = torch.empty((batch, c * d, h, w), dtype=torch.float32, device=features.device)
        with _timed("bev_scatter_fwd", n=n, c=c, out_elems=out.numel()):
            _C.check(_C.lib().toda_bev_scatter_fwd(_p(features), _p(coords), n, c, batch, d, h, w, _p(out), _stream()),
                     "toda_bev_scatter_fwd")
        ctx.save_for_backward(coords)
        ctx.dims = (n, c, batch, d, h, w)
        return out

    @staticmethod
    def backward(ctx, dout):
        (coords,) = ctx.saved_tensors
        n, c, batch, d, h, w = ctx.dims
        dout = dout.contiguous()
        df = torch.empty((n, c), dtype=torch.float32, device=dout.device)
        with _timed("bev_scatter_bwd", n=n, c=c):
            _C.check(_C.lib().toda_bev_scatter_bwd(_p(dout), _p(coords), n, c, batch, d, h, w, _p(df), _stream()),
                     "toda_bev_scatter_bwd")
        return df, None, None, None, None, None


def bev_scatter(features, coords, batch, d, h, w):
    """(B, C*D, H, W) dense BEV map; height_compression.py L20-25."""
    return _BEVScatter.apply(features, coords, batch, d, h, w)


class _GatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, rows, inverse_rows):
        x = _need(x.contiguous(), torch.float32, "features")
        n, c = rows.shape[0], x.shape[1]
        out = torch.empty((n, c), dtype=torch.float32, device=x.device)
        _C.check(_C.lib().toda_gather_rows(_p(x), _p(rows), n, c, _p(out), _stream()), "toda_gather_rows")
        ctx.save_for_backward(inverse_rows)
        return out

    @staticmethod
    def backward(ctx, dout):
        (inv,) = ctx.saved_tensors
        dout = dout.contiguous()
        n, c = inv.shape[0], dout.shape[1]
        dx = torch.empty((n, c), dtype=torch.float32, device=dout.device)
        _C.check(_C.lib().toda_gather_rows(_p(dout), _p(inv), n, c, _p(dx), _stream()), "toda_gather_rows")
        return dx, None, None


def permute_rows(x, rows, inverse_rows):
    """out[i] = x[rows[i]] for a permutation `rows` (inverse given, used by the backward)."""
    return _GatherRows.apply(x, rows, inverse_rows)
