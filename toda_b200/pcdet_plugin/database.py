"""pcdet's GT database (the object crops that gt_sampling pastes into frames), read once and held on the device.

Reads the on-disk format of OpenPCDet v0.5.2's DataBaseSampler (pcdet/datasets/augmentor/database_sampler.py, __init__,
filter_by_difficulty, filter_by_min_points, add_sampled_boxes_to_scene):
  - DB_INFO_PATH: pickles (under root_path) of {class name: [info, ...]}, info a dict with at least 'name', 'path',
    'box3d_lidar', 'num_points_in_gt', 'difficulty' and, with USE_SHARED_MEMORY, 'global_data_offset';
  - the object points: root_path / info['path'], float32 with NUM_POINT_FEATURES columns, or with USE_SHARED_MEMORY the
    rows global_data_offset of the float32 (R, NUM_POINT_FEATURES) array saved at root_path / DB_DATA_PATH[0];
  - PREPARE: filter_by_difficulty / filter_by_min_points in their config order; only the classes in class_names are kept.
`parse_database` does that on the host; `upload_database` puts every kept object's points into one float32 device buffer.
`load_database` caches the result per process, so a database is read and uploaded once.
"""
import os
import pickle

import numpy as np
import torch


def _get(cfg, key, default=None):
    return cfg.get(key, default) if hasattr(cfg, "get") else getattr(cfg, key, default)


class HostDatabase:
    """The filtered database on the host.  Per class (in class_names order): `infos` (the info dicts), `boxes` (M, C) in
    the stored dtype, `names`, and `first_row` / `num_rows` (int64) of each object's points in `points` (R, F) float32."""

    def __init__(self, class_names, infos, points, first_row, num_rows, num_point_features):
        self.class_names = list(class_names)
        self.infos = infos
        self.points = points
        self.first_row, self.num_rows = first_row, num_rows
        self.num_point_features = num_point_features
        self.boxes, self.names = {}, {}
        dtypes = set()
        for c in self.class_names:
            self.boxes[c] = (np.stack([np.asarray(i["box3d_lidar"]) for i in infos[c]]) if infos[c] else np.zeros((0, 7), np.float32))
            self.names[c] = np.array([i["name"] for i in infos[c]])
            if infos[c]:
                dtypes.add(self.boxes[c].dtype)
        if len(dtypes) > 1:
            raise ValueError(f"GT database: box3d_lidar is stored in more than one dtype ({sorted(map(str, dtypes))})")
        self.box_dtype = dtypes.pop() if dtypes else np.dtype(np.float32)


def _filter_by_difficulty(db_infos, removed_difficulty):
    return {key: [info for info in dinfos if info["difficulty"] not in removed_difficulty] for key, dinfos in db_infos.items()}


def _filter_by_min_points(db_infos, min_gt_points_list):
    for name_num in min_gt_points_list:
        name, min_num = name_num.split(":")
        min_num = int(min_num)
        if min_num > 0 and name in db_infos.keys():
            db_infos[name] = [info for info in db_infos[name] if info["num_points_in_gt"] >= min_num]
    return db_infos


_FILTERS = {"filter_by_difficulty": _filter_by_difficulty, "filter_by_min_points": _filter_by_min_points}


def parse_database(root_path, sampler_cfg, class_names):
    """Reads and filters the database as DataBaseSampler.__init__ does, and reads the kept objects' points."""
    for key in ("USE_ROAD_PLANE", "DATABASE_WITH_FAKELIDAR"):
        if _get(sampler_cfg, key, False):
            raise NotImplementedError(f"gt_sampling: {key} (KITTI only) is not supported on the device")
    num_feat = int(_get(sampler_cfg, "NUM_POINT_FEATURES"))
    db_infos = {c: [] for c in class_names}
    for db_info_path in _get(sampler_cfg, "DB_INFO_PATH"):
        with open(os.path.join(root_path, db_info_path), "rb") as f:
            infos = pickle.load(f)
        for c in class_names:
            db_infos[c].extend(infos[c])
    prepare = _get(sampler_cfg, "PREPARE", None) or {}
    for func_name, val in prepare.items():
        if func_name not in _FILTERS:
            raise NotImplementedError(f"gt_sampling: PREPARE step {func_name!r} is not supported")
        db_infos = _FILTERS[func_name](db_infos, val)
    shared = None
    if _get(sampler_cfg, "USE_SHARED_MEMORY", False):
        shared = np.load(os.path.join(root_path, _get(sampler_cfg, "DB_DATA_PATH")[0]), mmap_mode="r")
        if shared.dtype != np.float32 or shared.ndim != 2 or shared.shape[1] != num_feat:
            raise ValueError(f"gt_sampling: DB_DATA_PATH holds {shared.dtype} {shared.shape}, not float32 (R, {num_feat})")
    chunks, first_row, num_rows, row = [], {}, {}, 0
    for c in class_names:
        firsts, counts = [], []
        for info in db_infos[c]:
            if shared is not None:
                start, end = info["global_data_offset"]
                pts = np.asarray(shared[start:end], dtype=np.float32)
            else:
                pts = np.fromfile(os.path.join(root_path, info["path"]), dtype=np.float32).reshape([-1, num_feat])
            chunks.append(pts)
            firsts.append(row)
            counts.append(pts.shape[0])
            row += pts.shape[0]
        first_row[c] = np.array(firsts, np.int64)
        num_rows[c] = np.array(counts, np.int64)
    points = np.concatenate(chunks) if chunks else np.zeros((0, num_feat), np.float32)
    return HostDatabase(class_names, db_infos, np.ascontiguousarray(points, np.float32), first_row, num_rows, num_feat)


def upload_database(host_db, device):
    """The points of every kept object as one float32 (R, F) device tensor; host_db.bytes_uploaded records its size."""
    pts = torch.from_numpy(host_db.points).to(device)
    host_db.bytes_uploaded = pts.numel() * pts.element_size()
    return pts


_CACHE = {}


def load_database(root_path, sampler_cfg, class_names):
    """parse_database, cached per process (keyed by the paths, filters and classes)."""
    key = (os.path.abspath(str(root_path)), tuple(_get(sampler_cfg, "DB_INFO_PATH")), repr(_get(sampler_cfg, "PREPARE", None)),
           bool(_get(sampler_cfg, "USE_SHARED_MEMORY", False)), tuple(_get(sampler_cfg, "DB_DATA_PATH", None) or ()),
           int(_get(sampler_cfg, "NUM_POINT_FEATURES")), tuple(class_names))
    if key not in _CACHE:
        _CACHE[key] = {"host": parse_database(root_path, sampler_cfg, class_names), "device": {}}
    return _CACHE[key]


def device_points(entry, device):
    """The cached database's device buffer on `device`, uploaded on first use."""
    device = torch.device(device)
    if device not in entry["device"]:
        entry["device"][device] = upload_database(entry["host"], device)
    return entry["device"][device]
