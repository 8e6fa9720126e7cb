"""pcdet plugin surface: the cfg-driven module NAMEs of the hot path, backed by libtoda_b200.

Registries mirror pcdet's (`vfe.__all__` pcdet/models/backbones_3d/vfe/__init__.py L8-15,
`backbones_3d.__all__` backbones_3d/__init__.py L5-11, `map_to_bev.__all__` map_to_bev/__init__.py L5-9);
`register(pcdet_models)` overwrites those entries in an imported pcdet so that `build_network` picks these
classes up with unchanged YAML configs.
"""
import torch
import torch.nn as nn

from .. import ops
from ..spconv_compat import pytorch as _sp
from .backbones import make_backbones

_classes = make_backbones(_sp, _sp.bn_act_tensor, _sp.conv_bn_act_tensor, _sp.res_block_tensor)
VoxelBackBone8x = _classes["VoxelBackBone8x"]
VoxelResBackBone8x = _classes["VoxelResBackBone8x"]
SparseBasicBlock = _classes["SparseBasicBlock"]


def frame_offsets(batch_dict):
    """int32 (B+1) row offsets of the frames of batch_dict['points']: `point_frame_offsets` when present, otherwise found
    from the batch column, since collate_batch stores the frames back to back (dataset.py L173-178)."""
    offsets = batch_dict.get("point_frame_offsets")
    if offsets is None:
        points = batch_dict["points"]
        bidx = points[:, 0].contiguous()
        bounds = torch.arange(int(batch_dict["batch_size"]) + 1, device=points.device, dtype=torch.float32)
        offsets = torch.searchsorted(bidx, bounds).int()
    return offsets


class MeanVFE(nn.Module):
    """pcdet/models/backbones_3d/vfe/mean_vfe.py; constructor as detector3d_template.py L56-63 calls it.

    With the reference's `transform_points_to_voxels` processor the batch already holds voxels / voxel_coords /
    voxel_num_points and only the mean is computed.  With `transform_points_to_voxels_placeholder`
    (data_processor.py L105-113) the batch holds `points` [b,x,y,z,...] on the GPU and the hard voxelization
    runs here (K1), which is where the work belongs once it is a GPU kernel; the cap parameters then come
    from model_cfg (MAX_POINTS_PER_VOXEL, MAX_NUMBER_OF_VOXELS) since pcdet does not hand the data config to
    the VFE.
    """

    def __init__(self, model_cfg, num_point_features, voxel_size=None, point_cloud_range=None, grid_size=None, **kwargs):
        super().__init__()
        self.model_cfg = model_cfg
        self.num_point_features = num_point_features
        self.voxel_size = voxel_size
        self.point_cloud_range = point_cloud_range
        self.grid_size = grid_size

    def get_output_feature_dim(self):
        return self.num_point_features

    def _cfg(self, key, default=None):
        cfg = self.model_cfg
        val = cfg.get(key, default) if hasattr(cfg, "get") else getattr(cfg, key, default)
        if val is None:
            raise KeyError(f"MeanVFE needs model_cfg.{key} to voxelize on the GPU")
        return val

    def voxelize(self, batch_dict):
        points = batch_dict["points"]                       # (N, 1+F): [b, x, y, z, ...]
        offsets = frame_offsets(batch_dict)
        mode = "train" if self.training else "test"
        max_voxels = self._cfg("MAX_NUMBER_OF_VOXELS")
        max_voxels = max_voxels[mode] if hasattr(max_voxels, "__getitem__") and not isinstance(max_voxels, int) else max_voxels
        voxels, coords, num, _ = ops.voxelize(
            points.contiguous(), offsets, self.point_cloud_range, self.voxel_size, int(self._cfg("MAX_POINTS_PER_VOXEL")),
            int(max_voxels), num_features=self.num_point_features, xyz_col=1, feat_col=1, order=ops.ORDER_CANONICAL,
            grid=self.grid_size)
        batch_dict["voxels"], batch_dict["voxel_coords"], batch_dict["voxel_num_points"] = voxels, coords, num
        batch_dict["voxel_coords_canonical"] = True
        return batch_dict

    def forward(self, batch_dict, **kwargs):
        if "voxels" not in batch_dict:
            batch_dict = self.voxelize(batch_dict)
        batch_dict["voxel_features"] = ops.mean_vfe(batch_dict["voxels"], batch_dict["voxel_num_points"])
        return batch_dict


class DynamicMeanVFE(nn.Module):
    """pcdet/models/backbones_3d/vfe/dynamic_mean_vfe.py (OpenPCDet v0.5.2), without torch_scatter.

    Reads `points` [b, x, y, z, ...] (the `transform_points_to_voxels_placeholder` path) and voxelizes with no caps:
    every point inside [0, grid_size) on all three axes counts, and each voxel's feature is the mean of columns 1..F of
    its points (fp32 sum in ascending point order).  Differences from the reference, by design: rows come in canonical
    (b, z, y, x) order instead of sorted (b, x, y, z) keys (each row's values are the same), points with a NaN coordinate
    are dropped, and the voxel key has no int32 wrap.  Like the reference's forward, nothing here carries a gradient.
    """

    def __init__(self, model_cfg, num_point_features, voxel_size, grid_size, point_cloud_range, **kwargs):
        super().__init__()
        self.model_cfg = model_cfg
        self.num_point_features = num_point_features
        self.voxel_size = voxel_size
        self.grid_size = grid_size
        self.point_cloud_range = point_cloud_range

    def get_output_feature_dim(self):
        return self.num_point_features

    @torch.no_grad()
    def forward(self, batch_dict, **kwargs):
        features, coords, _ = ops.voxelize_dynamic(batch_dict["points"].contiguous(), frame_offsets(batch_dict),
                                                   self.point_cloud_range, self.voxel_size, grid=self.grid_size)
        batch_dict["voxel_features"], batch_dict["voxel_coords"] = features, coords
        batch_dict["voxel_coords_canonical"] = True
        return batch_dict


class HeightCompression(nn.Module):
    """pcdet/models/backbones_2d/map_to_bev/height_compression.py: one scatter kernel writes (B, C*D, H, W)."""

    def __init__(self, model_cfg, **kwargs):
        super().__init__()
        self.model_cfg = model_cfg
        self.num_bev_features = self.model_cfg.NUM_BEV_FEATURES

    def forward(self, batch_dict):
        t = batch_dict["encoded_spconv_tensor"]
        d, h, w = t.spatial_shape
        idx = t.indices if t.indices.dtype == torch.int32 else t.indices.int()
        batch_dict["spatial_features"] = ops.bev_scatter(t.features, idx.contiguous(), t.batch_size, d, h, w)
        batch_dict["spatial_features_stride"] = batch_dict["encoded_spconv_tensor_stride"]
        return batch_dict


VFE = {"MeanVFE": MeanVFE, "DynamicMeanVFE": DynamicMeanVFE}
BACKBONES_3D = {"VoxelBackBone8x": VoxelBackBone8x, "VoxelResBackBone8x": VoxelResBackBone8x}
MAP_TO_BEV = {"HeightCompression": HeightCompression}


def register(pcdet_models):
    """Overwrite the hot-path entries of an imported `pcdet.models` package's registries."""
    pcdet_models.backbones_3d.vfe.__all__.update(VFE)
    pcdet_models.backbones_3d.__all__.update(BACKBONES_3D)
    pcdet_models.backbones_2d.map_to_bev.__all__.update(MAP_TO_BEV)
