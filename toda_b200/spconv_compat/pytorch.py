"""`spconv.pytorch`-shaped surface on top of libtoda_b200 (the drop-in contract of SURVEY.md section 8b).

Exactly the names the reference touches: SparseConvTensor (features / indices / spatial_shape /
batch_size / dense() / replace_feature()), SubMConv3d, SparseConv3d, SparseInverseConv3d, SparseSequential,
SparseModule and conv.SparseConvolution (pcdet/utils/spconv_utils.py L3-6, L19, L29-31;
pcdet/models/backbones_3d/spconv_backbone.py L12-21, L30, L38-45, L141-146; height_compression.py L21).

Row order: a SparseConvTensor keeps the caller's row order until its first convolution; convolution
outputs are in canonical (b,z,y,x) order with their own consistent `indices` (spconv leaves the order of
SparseConv3d outputs implementation-defined; for SubMConv3d it preserves the input order, which coincides
whenever the input is canonical, e.g. when it comes from toda_b200's voxelizer in canonical order).
"""
import math
from collections import OrderedDict

import numpy as np
import torch
import torch.nn as nn

from .. import ops

_precision = ops.CONV_FP32
# BatchNorm modules SparseSequential runs on libtoda_b200 (nn.SyncBatchNorm: what convert_sync_batchnorm makes of the former)
_FUSED_BN = (nn.BatchNorm1d, nn.SyncBatchNorm)


def set_conv_precision(p):
    """'fp32' (FFMA, parity path), 'bf16' (tcgen05 tensor cores, bf16 operands, fp32 accumulate) or 'bf16x3' (the same
    tensor-core kernels on split operands, three launches per product: fp32-class accuracy, rtol 1e-4 vs the oracle)."""
    global _precision
    _precision = {"fp32": ops.CONV_FP32, "bf16": ops.CONV_BF16, "bf16x3": ops.CONV_BF16X3}[p] if isinstance(p, str) else int(p)


def get_conv_precision():
    return _precision


def _triple(v):
    if isinstance(v, (list, tuple)):
        assert len(v) == 3
        return [int(x) for x in v]
    return [int(v)] * 3


class SparseConvTensor:
    def __init__(self, features, indices, spatial_shape, batch_size, grid=None, voxel_num=None, indice_dict=None,
                 benchmark=False, _index=None, _features_bf16=None, _bn_sums=None):
        self.features = features
        self.indices = indices
        self.spatial_shape = [int(s) for s in spatial_shape]
        self.batch_size = int(batch_size)
        self.indice_dict = indice_dict if indice_dict is not None else {}
        self.grid = grid
        self.voxel_num = voxel_num
        self.benchmark = benchmark
        self._index = _index          # ops.OccupancyIndex when rows are in canonical order
        self._features_bf16 = _features_bf16   # bf16 copy of `features` written by the fused BN pass (tensor-core operand)
        self._bn_sums = _bn_sums               # per-channel (sum, sum^2) of `features` from the conv epilogue, for the next BN

    def replace_feature(self, feature, _features_bf16=None):
        return SparseConvTensor(feature, self.indices, self.spatial_shape, self.batch_size, self.grid, self.voxel_num,
                                self.indice_dict, self.benchmark, self._index, _features_bf16)

    @property
    def spatial_size(self):
        return int(np.prod(self.spatial_shape))

    def canonical(self, assume_canonical=False):
        """This tensor with rows in (b,z,y,x) order and a live occupancy index."""
        if self._index is not None:
            return self
        indices = self.indices
        if indices.dtype != torch.int32:
            indices = indices.int()
        indices = indices.contiguous()
        n = indices.shape[0]
        index = ops.OccupancyIndex(self.batch_size, self.spatial_shape, indices.device, "level")
        index.insert(indices)
        coords = index.build(n)
        if index.n != n:
            raise ValueError(f"SparseConvTensor indices hold {n - index.n} duplicate or out-of-range coordinates")
        if assume_canonical or bool(torch.equal(coords, indices)):
            feats = self.features
        else:
            rows = index.rows(indices)                       # canonical row of every input row
            inv = torch.empty_like(rows)
            inv[rows.long()] = torch.arange(n, dtype=torch.int32, device=rows.device)
            feats = ops.permute_rows(self.features, inv, rows)
        return SparseConvTensor(feats, coords, self.spatial_shape, self.batch_size, self.grid, self.voxel_num,
                                self.indice_dict, self.benchmark, index)

    def dense(self, channels_first=True):
        """zeros (B,C,D,H,W) with features scattered in (Appendix C.3)."""
        idx = self.indices if self.indices.dtype == torch.int32 else self.indices.int()
        d, h, w = self.spatial_shape
        c = self.features.shape[1]
        out = ops.bev_scatter(self.features, idx.contiguous(), self.batch_size, d, h, w).view(self.batch_size, c, d, h, w)
        if not channels_first:
            return out.permute(0, 2, 3, 4, 1).contiguous()
        return out


def bn_act_tensor(x, bn, residual, relu):
    """Fused BatchNorm1d (+residual) (+ReLU) on a SparseConvTensor; in bf16 mode the same pass also writes the bf16
    copy that the next convolution gathers from."""
    if _precision == ops.CONV_BF16:
        a, ab = ops.bn_act(x.features, bn, residual, relu, want_bf16=True, sums=x._bn_sums)
        return x.replace_feature(a, ab)
    return x.replace_feature(ops.bn_act(x.features, bn, residual, relu, sums=x._bn_sums))


def conv_bn_act_tensor(x, conv, bn, residual, relu):
    """bn_act_tensor(conv(x), bn, residual, relu) as one autograd node (ops.conv_bn_act): same kernels, half the host work."""
    x = x.canonical()
    rb, index_out = conv._rulebook(x)
    bf16 = _precision == ops.CONV_BF16
    a, ab = ops.conv_bn_act(x.features, conv.weight, conv.bias, rb, _precision, bn, residual, relu, x._features_bf16, bf16)
    return SparseConvTensor(a, rb.out_coords, rb.out_shape, x.batch_size, x.grid, x.voxel_num, x.indice_dict, x.benchmark,
                            index_out, ab)


def res_block_tensor(x, conv1, bn1, conv2, bn2):
    """SparseBasicBlock (two SubMConv3d sharing one rulebook, BN, residual, ReLU) as one autograd node (ops.res_block)."""
    x = x.canonical()
    rb, index_out = conv1._rulebook(x)
    rb2, _ = conv2._rulebook(x)
    assert rb2 is rb, "SparseBasicBlock: both convolutions must share one indice_key"
    bf16 = _precision == ops.CONV_BF16
    a, ab = ops.res_block(x.features, x._features_bf16, conv1.weight, conv1.bias, bn1, conv2.weight, conv2.bias, bn2, rb,
                          _precision, bf16)
    return SparseConvTensor(a, rb.out_coords, rb.out_shape, x.batch_size, x.grid, x.voxel_num, x.indice_dict, x.benchmark,
                            index_out, ab)


class SparseModule(nn.Module):
    """Marker base: SparseSequential hands the whole SparseConvTensor to these."""
    pass


class SparseSequential(SparseModule):
    def __init__(self, *args, **kwargs):
        super().__init__()
        if len(args) == 1 and isinstance(args[0], OrderedDict):
            for key, module in args[0].items():
                self.add_module(key, module)
        else:
            for i, module in enumerate(args):
                self.add_module(str(i), module)
        for name, module in kwargs.items():
            self.add_module(name, module)

    def __getitem__(self, idx):
        return list(self._modules.values())[idx]

    def __len__(self):
        return len(self._modules)

    def add(self, module, name=None):
        self.add_module(name if name is not None else str(len(self._modules)), module)

    def forward(self, x):
        mods = list(self._modules.values())
        i = 0
        while i < len(mods):
            m = mods[i]
            if (isinstance(m, SparseConvolution) and isinstance(x, SparseConvTensor) and i + 1 < len(mods)
                    and type(mods[i + 1]) in _FUSED_BN and mods[i + 1].affine and mods[i + 1].track_running_stats
                    and x.features.is_cuda and x.indices.shape[0] > 0):
                # conv + BatchNorm1d / SyncBatchNorm [+ ReLU]: one fused autograd node
                relu = i + 2 < len(mods) and type(mods[i + 2]) is nn.ReLU
                x = conv_bn_act_tensor(x, m, mods[i + 1], None, relu)
                i += 3 if relu else 2
            elif isinstance(m, SparseModule):
                x = m(x)
                i += 1
            elif isinstance(x, SparseConvTensor):
                if x.indices.shape[0] == 0 and ops.sync_group(m) is not None and x.features.is_cuda:
                    # a synchronized BatchNorm on an empty tensor: this rank joins its peers' collectives (forward and
                    # backward) with a zero contribution, and takes the running statistics of the union batch
                    relu = i + 1 < len(mods) and type(mods[i + 1]) is nn.ReLU
                    x = bn_act_tensor(x, m, None, relu)
                    i += 2 if relu else 1
                    continue
                if x.indices.shape[0] == 0:
                    # spconv skips the feature modules on an empty tensor; a training BatchNorm1d still counts the batch
                    # (torch.nn.BatchNorm1d on zero rows: running statistics unchanged, num_batches_tracked + 1)
                    if isinstance(m, nn.modules.batchnorm._BatchNorm) and m.training and m.num_batches_tracked is not None:
                        m.num_batches_tracked += 1
                    i += 1
                    continue
                # BatchNorm1d / SyncBatchNorm [+ ReLU] after a conv: one fused pass of libtoda_b200 instead of ATen's
                if type(m) in _FUSED_BN and m.affine and m.track_running_stats and x.features.is_cuda:
                    relu = i + 1 < len(mods) and type(mods[i + 1]) is nn.ReLU
                    x = bn_act_tensor(x, m, None, relu)
                    i += 2 if relu else 1
                else:
                    x = x.replace_feature(m(x.features))
                    i += 1
            else:
                x = m(x)
                i += 1
        return x


class SparseConvolution(SparseModule):
    """weight: (Cout, kz, ky, kx, Cin) (accepted by detector3d_template.py L341-348); bias: (Cout,)."""

    def __init__(self, ndim, in_channels, out_channels, kernel_size=3, stride=1, padding=0, dilation=1, groups=1,
                 bias=True, subm=False, output_padding=0, transposed=False, inverse=False, indice_key=None, algo=None,
                 fp32_accum=None, name=None):
        super().__init__()
        if ndim != 3 or groups != 1 or transposed or inverse or _triple(dilation) != [1, 1, 1]:
            raise NotImplementedError("toda_b200 supports 3-D, dense-group, dilation-1 sparse convolutions")
        self.ndim = ndim
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.kernel_size = _triple(kernel_size)
        self.stride = _triple(stride)
        self.padding = _triple(padding)
        self.dilation = [1, 1, 1]
        self.subm = subm
        self.indice_key = indice_key
        self.weight = nn.Parameter(torch.empty(out_channels, *self.kernel_size, in_channels))
        if bias:
            self.bias = nn.Parameter(torch.empty(out_channels))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            fan_in = self.in_channels * int(np.prod(self.kernel_size))
            bound = 1 / math.sqrt(fan_in)
            nn.init.uniform_(self.bias, -bound, bound)

    def extra_repr(self):
        return (f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, stride={self.stride}, "
                f"padding={self.padding}, subm={self.subm}, indice_key={self.indice_key}")

    def _rulebook(self, x):
        key = self.indice_key
        hit = x.indice_dict.get(key) if key is not None else None
        if hit is not None:
            rb, index_out = hit
            geom_ok = (rb.subm == self.subm and rb.ksize == self.kernel_size and rb.in_shape == x.spatial_shape
                       and rb.n_in == x.features.shape[0] and (self.subm or (rb.stride == self.stride and rb.padding == self.padding)))
            if geom_ok:
                return rb, index_out
        if self.subm:
            rb = ops.rulebook_subm(x._index, self.kernel_size, channels=max(self.in_channels, self.out_channels))
            index_out = x._index
        else:
            rb, index_out = ops.rulebook_sparse(x._index, self.kernel_size, self.stride, self.padding, ("out", str(key)),
                                                cin=self.in_channels, cout=self.out_channels)
        if key is not None:
            x.indice_dict[key] = (rb, index_out)
        return rb, index_out

    def forward(self, x):
        assert isinstance(x, SparseConvTensor)
        x = x.canonical()
        rb, index_out = self._rulebook(x)
        # in tensor-core mode the epilogue also accumulates the statistics a following BatchNorm needs (train mode)
        want_stats = _precision in (ops.CONV_BF16, ops.CONV_BF16X3) and self.training and torch.is_grad_enabled()
        if want_stats:
            y, sums = ops.sparse_conv(x.features, self.weight, self.bias, rb, _precision, x._features_bf16, want_stats=True)
        else:
            y, sums = ops.sparse_conv(x.features, self.weight, self.bias, rb, _precision, x._features_bf16), None
        return SparseConvTensor(y, rb.out_coords, rb.out_shape, x.batch_size, x.grid, x.voxel_num, x.indice_dict,
                                x.benchmark, index_out, None, sums)


class GeometryPlan:
    """Everything about a sparse tensor chain that depends on coordinates only: the canonical input index and the
    rulebook of every `indice_key`.  Built ahead of time (e.g. on a side stream while the previous batch trains, see
    toda_b200.pipeline) it makes the forward pass free of index kernels and host synchronisation."""

    def __init__(self, index, coords, spatial_shape, batch_size, indice_dict):
        self.index, self.coords, self.spatial_shape, self.batch_size = index, coords, spatial_shape, batch_size
        self.indice_dict = indice_dict

    def tensors(self):
        out = [self.coords, self.index.frame_counts]
        for rb, index_out in self.indice_dict.values():
            out += [rb.out_coords, rb.nbr_fwd]
            if rb.tile_masks is not None:
                out.append(rb.tile_masks)
            if rb.nbr_bwd is not None:
                out.append(rb.nbr_bwd)
            if index_out.frame_counts is not None:
                out.append(index_out.frame_counts)
            if rb.dgrad_order is not None:
                out += [rb.dgrad_order, rb.nbr_bwd_sorted, rb.dgrad_tile_masks]
            for pl in (rb.plan, rb.dgrad_plan):
                if pl is not None:
                    out += pl.tensors()
        return [t for t in out if t is not None]

    def sparse_tensor(self, features, features_bf16=None):
        return SparseConvTensor(features, self.coords, self.spatial_shape, self.batch_size, indice_dict=self.indice_dict,
                                _index=self.index, _features_bf16=features_bf16)


class _GeometryCursor:
    """Stand-in for a SparseConvTensor while planning: coordinates and index, no features."""

    class _Rows:
        def __init__(self, n):
            self.shape = (n,)

    def __init__(self, index, coords, spatial_shape, indice_dict):
        self._index, self.indices, self.spatial_shape, self.indice_dict = index, coords, spatial_shape, indice_dict
        self.features = self._Rows(coords.shape[0])


def plan_geometry(convs, indices, spatial_shape, batch_size, assume_canonical=False):
    """Rulebooks for `convs` (SparseConvolution modules in execution order) applied as a chain to a tensor with
    `indices` (N,4) [b,z,y,x].  Needs canonical (b,z,y,x) row order (what toda_b200's voxelizer emits in canonical
    mode): a plan cannot permute features it has not seen."""
    x = SparseConvTensor(None, indices, spatial_shape, batch_size)
    if not assume_canonical:
        idx = indices.int().contiguous()
        index = ops.OccupancyIndex(batch_size, x.spatial_shape, idx.device, "level")
        index.insert(idx)
        coords = index.build(idx.shape[0])
        if index.n != idx.shape[0] or not bool(torch.equal(coords, idx)):
            raise ValueError("plan_geometry needs unique coordinates in canonical (b,z,y,x) order")
    else:
        idx = indices if indices.dtype == torch.int32 else indices.int()
        idx = idx.contiguous()
        index = ops.OccupancyIndex(batch_size, x.spatial_shape, idx.device, "level")
        index.insert(idx)
        coords = index.build(idx.shape[0], known_n=idx.shape[0])
    indice_dict = {}
    plan = GeometryPlan(index, coords, x.spatial_shape, x.batch_size, indice_dict)
    cur = _GeometryCursor(index, coords, x.spatial_shape, indice_dict)
    for m in convs:
        if m.indice_key is None:
            raise ValueError("plan_geometry needs an indice_key on every convolution")
        rb, index_out = m._rulebook(cur)
        if not m.subm:
            cur = _GeometryCursor(index_out, rb.out_coords, rb.out_shape, indice_dict)
    return plan


class SubMConv3d(SparseConvolution):
    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 indice_key=None, algo=None, fp32_accum=None, name=None):
        super().__init__(3, in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias, True,
                         indice_key=indice_key)
        if self.stride != [1, 1, 1]:
            raise NotImplementedError("SubMConv3d requires stride 1")


class SparseConv3d(SparseConvolution):
    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1, bias=True,
                 indice_key=None, algo=None, fp32_accum=None, name=None):
        super().__init__(3, in_channels, out_channels, kernel_size, stride, padding, dilation, groups, bias, False,
                         indice_key=indice_key)


class SparseInverseConv3d(SparseModule):
    """Named by post_act_block's unused 'inverseconv' branch only (spconv_backbone.py L16-17); not on the hot path."""

    def __init__(self, *a, **kw):
        super().__init__()
        raise NotImplementedError("SparseInverseConv3d is outside the hot path (SURVEY.md section 8b)")
