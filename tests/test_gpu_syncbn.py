"""BatchNorm synchronized across processes (torch.nn.SyncBatchNorm) on the fused sparse-conv layers.

  1. One GPU, no collective: the rows of a level are split into shards (one of them empty), each shard runs the local
     phase of the product (ops._layer_forward_phases / _layer_backward_phases, fused and stepwise), the shards' buffers are
     summed in torch as a stand-in for the all-reduce, and each shard finishes.  The concatenated outputs, dx, the summed
     dw / dgamma / dbeta and the running statistics must match a float64 BatchNorm over the union of the shards, with the
     tolerances and bf16 rounding allowances of tests/test_gpu_layers.py (RefLayer).  Shards are frames: a SubM
     convolution never mixes frames, so the union's conv output is the shards' outputs concatenated in frame order.
  2. World size 1: the split phases with the local buffers passed through equal toda_layer_fwd / toda_layer_bwd bit for
     bit, and a convert_sync_batchnorm'd backbone gives a bit-identical train step.
  3. Two processes on two GPUs (skipped with fewer): rank r runs frame r through the converted VoxelResBackBone8x and
     HeightCompression, compared with one process running both frames as one batch.

Tolerance of the two-process bf16 case: each rank's bf16 convolutions see the other rank's statistics only through the
BatchNorm coefficients, so the two runs differ where a value near a bf16 rounding midpoint rounds the other way
(fp32-accumulated sums in a different order).  Over the 21 layers of the backbone such flips accumulate like the bf16
error itself; a rel-L2 bound of 2e-2 is used, below the 5e-2 ceiling and well above what one flipped term per layer gives.
"""
import datetime
import os
import tempfile

import numpy as np
import pytest
import torch
import torch.distributed as dist

from tests import parity_utils as PU
from tests import test_gpu_layers as TL

pytestmark = pytest.mark.gpu
DEV = "cuda"
PRECISIONS = ("fp32", "bf16", "bf16x3")


def _ops():
    from toda_b200 import ops
    return ops


def _drive_in_lockstep(gens):
    """Runs the phase generators of all shards side by side; the buffers each phase yields are summed across the shards
    (what dist.all_reduce(SUM) does across ranks).  -> the generators' results."""
    results = [None] * len(gens)
    bufs = [next(g) for g in gens]
    while True:
        total = torch.stack(bufs).sum(0)
        nxt = []
        for i, (g, b) in enumerate(zip(gens, bufs)):
            b.copy_(total)
            try:
                nxt.append(g.send(None))
            except StopIteration as stop:
                results[i] = stop.value
        if all(r is not None for r in results):
            return results
        assert all(r is None for r in results), "shards disagree on the number of collectives"
        bufs = nxt


def _random_frames(sizes, shape, seed):
    """Canonical (b,z,y,x) coordinates of len(sizes) frames with sizes[f] distinct random voxels each (numpy)."""
    rng = np.random.default_rng(seed)
    cells = shape[0] * shape[1] * shape[2]
    out = []
    for f, n in enumerate(sizes):
        lin = np.sort(rng.choice(cells, size=n, replace=False))
        z, rem = np.divmod(lin, shape[1] * shape[2])
        y, x = np.divmod(rem, shape[2])
        out.append(np.stack([np.full(n, f), z, y, x], 1).astype(np.int32))
    return np.concatenate(out, 0)


class Split:
    """A union SubM geometry (TL.Geo, oracle pairs) over several frames and the product's rulebook of each frame alone."""

    def __init__(self, coords, shape, batch, tag):
        ops = _ops()
        self.shape, self.batch = list(shape), batch
        index = ops.OccupancyIndex(batch, shape, torch.device(DEV, 0), (tag, "union"))
        index.insert(torch.from_numpy(coords).to(DEV))
        index.build(coords.shape[0], known_n=coords.shape[0])
        self.geo = TL._subm_geo(index, coords, shape)
        self.rows, self.rbs, self._indices = [], [], []
        for f in range(batch):
            sel = np.nonzero(coords[:, 0] == f)[0]
            self.rows.append(torch.from_numpy(sel).to(DEV))
            c = coords[sel].copy()
            c[:, 0] = 0
            idx = ops.OccupancyIndex(1, shape, torch.device(DEV, 0), (tag, f))
            idx.insert(torch.from_numpy(c).to(DEV))
            idx.build(c.shape[0], known_n=c.shape[0])
            self._indices.append(idx)
            self.rbs.append(ops.rulebook_subm(idx, [3, 3, 3]))


def _split_small(sizes, seed):
    shape = [40, 50, 60]
    return Split(_random_frames(sizes, shape, seed), shape, len(sizes), ("syncbn_small", seed))


@pytest.fixture(scope="module")
def full_split():
    """The two full-size nuScenes-shaped frames of tests/test_gpu_layers.py (level 1) plus an empty third frame."""
    from toda_b200 import synth
    ops = _ops()
    cfg = synth.CONFIGS["nus_0075"]
    frames, collated = synth.make_batch("nus_0075", 2)
    offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(DEV)
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    _, coords, _, _ = ops.voxelize(torch.from_numpy(collated).to(DEV), offs, cfg["pc_range"], cfg["voxel_size"], 10, 120000,
                                   xyz_col=1, feat_col=1, num_features=5, order=ops.ORDER_CANONICAL, grid=grid)
    c = coords.cpu().numpy()
    c = np.concatenate([c[c[:, 0] == 0], c[c[:, 0] == 1]], 0)
    c[:, 0] = np.where(c[:, 0] == 1, 2, 0)              # frames 0 and 2 full, frame 1 empty
    shape = [int(grid[2]) + 1, int(grid[1]), int(grid[0])]
    return Split(c, shape, 3, "syncbn_full")


def _bns(c, n, momentum, seed):
    """n identical BatchNorm1d replicas (one per shard / rank) -> (replicas, the state before the step)."""
    bn = TL.make_bn(c, momentum, seed)
    reps = []
    for _ in range(n):
        r = torch.nn.BatchNorm1d(c, eps=bn.eps, momentum=bn.momentum).to(DEV)
        r.load_state_dict(bn.state_dict())
        reps.append(r)
    return reps, {k: v.clone() for k, v in bn.state_dict().items()}


def _layer_shards(split, x, w, b, prec, bns, g, residual=None, relu=True, stepwise=False, addend_of=None):
    """One conv -> BN (+residual) -> ReLU layer on every shard through the phase generators, forward and backward.
    -> (a per shard, saved per shard, backward results per shard)."""
    ops = _ops()
    p = TL._prec(prec)
    if stepwise:
        ops.profile_begin()      # a profile pass routes the layer through the stepwise kernels
    try:
        fw = _drive_in_lockstep([
            ops._layer_forward_phases(x[r], None, w, b, rb, p, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps,
                                      bn.momentum, residual[i] if residual is not None else None, relu, False)
            for i, (rb, r, bn) in enumerate(zip(split.rbs, split.rows, bns))])
        for bn in bns:
            bn.num_batches_tracked += 1
        bw = _drive_in_lockstep([
            ops._layer_backward_phases(g[r].contiguous(), saved, rb, p, relu, residual is not None, b is not None, True, True,
                                       addend_of[i] if addend_of is not None else None)
            for i, (rb, r, (_, _, saved)) in enumerate(zip(split.rbs, split.rows, fw))])
    finally:
        if stepwise:
            ops.profile_end()
    return [f[0] for f in fw], [f[2] for f in fw], bw


def _union(split, parts, width):
    out = torch.zeros((split.geo.n_out, width), dtype=parts[0].dtype, device=DEV) if parts else None
    for r, t in zip(split.rows, parts):
        out[r] = t
    return out


def _check_running(bns, ref_bn, tag, tols):
    for bn in bns[1:]:
        assert torch.equal(bn.running_mean, bns[0].running_mean) and torch.equal(bn.running_var, bns[0].running_var)
    for bn in bns:
        assert int(bn.num_batches_tracked) == 1
    TL.check(bns[0].running_mean, ref_bn.running_mean, *tols, what=f"running_mean {tag}")
    TL.check(bns[0].running_var, ref_bn.running_var, *tols, what=f"running_var {tag}")


def run_sharded_layer(split, cin, cout, prec, seed, tag, stepwise=False):
    x, w, _ = TL.make_operands(split.geo, cin, cout, prec, seed, bias=False)
    b = torch.randn((cout,), device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 3)) * 0.1
    bns, before = _bns(cout, len(split.rbs), 0.5, seed + 1)
    g = torch.randn((split.geo.n_out, cout), device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed + 2))
    a_s, _, bw = _layer_shards(split, x, w, b, prec, bns, g, stepwise=stepwise)
    a = _union(split, a_s, cout)
    ref_bn = torch.nn.BatchNorm1d(cout, eps=1e-3, momentum=0.5).to(DEV)
    ref_bn.load_state_dict(before)
    ref = TL.RefLayer(x, w, b, split.geo, ref_bn, True, mask=a > 0)
    TL.check_masks(a, ref.z, f"sharded mask {tag}")
    TL.check(a, ref.a, what=f"sharded a {tag}")
    _check_running(bns, ref, tag, (PU.RTOL, 1e-5))
    rd, rw = TL._rounders(cin, cout, 27, prec)
    r = ref.backward(g, prec, rd, rw)
    rtol, atol = TL.bwd_tols(prec)
    dx = _union(split, [o[0] for o in bw], cin)
    TL.check(dx, r["dx"], rtol, atol, what=f"sharded dx {tag}", allow=r["fdx"])
    TL.check(sum(o[1] for o in bw), r["dw"], rtol, atol, what=f"sharded sum dw {tag}", allow=r["fdw"])
    TL.check(sum(o[3] for o in bw), r["dgamma"], rtol, atol, what=f"sharded sum dgamma {tag}")
    TL.check(sum(o[4] for o in bw), r["dbeta"], rtol, atol, what=f"sharded sum dbeta {tag}")
    TL.check_zero_bias_grad(sum(o[2] for o in bw), r["dy"], rtol, what=f"sharded sum db {tag}")


# ---------------------------------------------------------------------------------------------- 1. phases on one GPU
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("stepwise", [False, True], ids=["fused", "stepwise"])
@pytest.mark.parametrize("cout", [6, 12, 16, 32, 64, 128])
def test_sharded_layer_ragged_vs_fp64(cout, stepwise, prec):
    """Three shards of 1500, 0 and 2201 rows (ragged last tiles, one empty rank) of one layer, C = 6 / 12 (scalar BatchNorm
    kernels) to 128."""
    split = _split_small([1500, 0, 2201], seed=cout)
    run_sharded_layer(split, 16, cout, prec, seed=10 * cout + 1, tag=f"ragged C={cout} {'stepwise' if stepwise else 'fused'} {prec}")


@pytest.mark.parametrize("prec", PRECISIONS)
def test_sharded_layer_full_size_vs_fp64(full_split, prec):
    """Two full-size frames and an empty one, level 1 (SubM 3x3x3, 16 -> 64 channels)."""
    run_sharded_layer(full_split, 16, 64, prec, seed=77, tag=f"full {prec}")


@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("c", [16, 32])
def test_sharded_res_block_vs_fp64(c, prec):
    """SparseBasicBlock (the two layers of ops._ResBlock, residual-branch gradient in conv1's dgrad) on three shards."""
    split = _split_small([2000, 0, 1300], seed=500 + c)
    blk = TL._block(c, prec, seed=c)
    blk.train()
    before = TL._bn_states(blk)
    n = len(split.rbs)
    bn1s, bn2s = [], []
    for _ in range(n):
        for lst, bn in ((bn1s, blk.bn1), (bn2s, blk.bn2)):
            r = torch.nn.BatchNorm1d(c, eps=bn.eps, momentum=bn.momentum).to(DEV)
            r.load_state_dict(bn.state_dict())
            r.weight.requires_grad_(False)
            r.bias.requires_grad_(False)
            lst.append(r)
    x, _ = TL._canonical_tensor(split.geo, c, prec, seed=c + 1)
    g = torch.randn((split.geo.n_out, c), device=DEV, generator=torch.Generator(device=DEV).manual_seed(c + 2))
    ops = _ops()
    p = TL._prec(prec)
    w1, b1, w2, b2 = (t.detach() for t in (blk.conv1.weight, blk.conv1.bias, blk.conv2.weight, blk.conv2.bias))
    xs = [x[r].contiguous() for r in split.rows]
    f1 = _drive_in_lockstep([ops._layer_forward_phases(xs[i], None, w1, b1, rb, p, bn.weight, bn.bias, bn.running_mean,
                                                       bn.running_var, bn.eps, bn.momentum, None, True, False)
                             for i, (rb, bn) in enumerate(zip(split.rbs, bn1s))])
    f2 = _drive_in_lockstep([ops._layer_forward_phases(f1[i][0], None, w2, b2, rb, p, bn.weight, bn.bias, bn.running_mean,
                                                       bn.running_var, bn.eps, bn.momentum, xs[i], True, False)
                             for i, (rb, bn) in enumerate(zip(split.rbs, bn2s))])
    for bn in bn1s + bn2s:
        bn.num_batches_tracked += 1
    b2r = _drive_in_lockstep([ops._layer_backward_phases(g[r].contiguous(), f2[i][2], rb, p, True, True, True, True, True)
                              for i, (rb, r) in enumerate(zip(split.rbs, split.rows))])
    b1r = _drive_in_lockstep([ops._layer_backward_phases(b2r[i][0], f1[i][2], rb, p, True, False, True, True, True,
                                                         addend=b2r[i][5])
                              for i, rb in enumerate(split.rbs)])
    h = _union(split, [f[0] for f in f1], c)
    out = _union(split, [f[0] for f in f2], c)
    with torch.no_grad():
        for bn, reps in ((blk.bn1, bn1s), (blk.bn2, bn2s)):
            for r in reps[1:]:
                assert torch.equal(r.running_mean, reps[0].running_mean) and torch.equal(r.running_var, reps[0].running_var)
            bn.running_mean.copy_(reps[0].running_mean)
            bn.running_var.copy_(reps[0].running_var)
    for conv, bn, res in ((blk.conv1, blk.bn1, b1r), (blk.conv2, blk.bn2, b2r)):
        conv.weight.grad = sum(o[1] for o in res)
        conv.bias.grad = sum(o[2] for o in res)
        bn.weight.grad = sum(o[3] for o in res)
        bn.bias.grad = sum(o[4] for o in res)
    xx = x.clone()
    xx.grad = _union(split, [o[0] for o in b1r], c)
    l1, l2 = TL._ref_block(blk, before, x, split.geo, True, h, out > 0, prec)
    r1, r2 = TL._block_backward(l1, l2, g, c, prec)
    TL._compare_block(blk, xx, out, h, l1, l2, r1, r2, True, prec, f"sharded block C={c} {prec}")


# ---------------------------------------------------------------------------------------------- 2. world size 1
@pytest.mark.parametrize("prec", PRECISIONS)
@pytest.mark.parametrize("cout", [12, 64])
@pytest.mark.parametrize("stepwise", [False, True], ids=["fused", "stepwise"])
def test_split_phases_equal_single_call_bitwise(stepwise, cout, prec):
    """stats + apply and reduce + finish with the local buffers passed through unreduced compute exactly what
    toda_layer_fwd / toda_layer_bwd (and their stepwise counterparts) compute.  The tensor-core epilogue accumulates its
    statistics with fp64 atomics, whose order is not fixed; where two runs of the single call differ, the comparison is
    against the single call's own run-to-run spread instead."""
    ops = _ops()
    split = _split_small([3001], seed=900 + cout)
    rb = split.rbs[0]
    p = TL._prec(prec)
    x, w, _ = TL.make_operands(split.geo, 16, cout, prec, seed=cout)
    g = torch.randn((rb.n_out, cout), device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    bf16 = prec == "bf16"

    def run(sync):
        bn = TL.make_bn(cout, 0.5, 4)
        if stepwise:
            ops.profile_begin()
        try:
            if sync:
                (a, ab, saved), = _drive_in_lockstep([ops._layer_forward_phases(
                    x, None, w, None, rb, p, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps, bn.momentum, None, True,
                    bf16)])
                back, = _drive_in_lockstep([ops._layer_backward_phases(g, saved, rb, p, True, False, False, True, True)])
            else:
                a, ab, saved = ops._layer_forward(x, None, w, None, rb, p, bn.weight, bn.bias, bn.running_mean, bn.running_var,
                                                  bn.eps, bn.momentum, True, None, True, bf16)
                back = ops._layer_backward(g, saved, rb, p, True, True, False, False, True, True)
        finally:
            if stepwise:
                ops.profile_end()
        return [a, ab, bn.running_mean, bn.running_var, saved[6], saved[7]] + [back[i] for i in (0, 1, 3, 4)]

    names = ["a", "a_bf16", "running_mean", "running_var", "mean", "rstd", "dx", "dw", "dgamma", "dbeta"]
    one, two, split_run = run(False), run(False), run(True)
    for nm, u, v, s in zip(names, one, two, split_run):
        if u is None:
            assert s is None, nm
            continue
        if torch.equal(u, v):
            assert torch.equal(u, s), f"{nm}: split phases differ from the single call"
        else:
            spread = float((u.double() - v.double()).abs().max())
            err = float((u.double() - s.double()).abs().max())
            print(f"{nm}: the single call is not run-to-run deterministic here (spread {spread:.3e}); split error {err:.3e}")
            assert err <= 4 * spread, nm


def _backbone_step(net, vf, coords, prec, seed):
    import toda_b200.pcdet_plugin as P
    from toda_b200.spconv_compat import pytorch as G
    hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
    G.set_conv_precision(prec)
    try:
        v = vf.clone().requires_grad_(True)
        sf = hc(net({"voxel_features": v, "voxel_coords": coords, "batch_size": 2}))["spatial_features"]
        cot = torch.randn(sf.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed))
        (sf * cot).sum().backward()
    finally:
        G.set_conv_precision("fp32")
    return sf.detach(), v.grad


def _small_input(seed, n=6000, batch=2):
    shape = [41, 200, 176]
    coords = _random_frames([n // batch] * batch, shape, seed)
    vf = torch.randn((coords.shape[0], 5), device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed))
    return vf, torch.from_numpy(coords).to(DEV), [176, 200, 40]


@pytest.mark.parametrize("prec", ["fp32"])
def test_world_size_one_backbone_bitwise(prec, tmp_path):
    """convert_sync_batchnorm'd VoxelResBackBone8x, with torch.distributed initialized on one rank: no collective, and
    outputs, gradients and running statistics bit-identical to the BatchNorm1d backbone.  Eval mode issues no
    collective either.  fp32 only: the tensor-core epilogue's fp64 atomics make two bf16 runs of the same backbone differ
    in the last bits."""
    import toda_b200.pcdet_plugin as P
    vf, coords, grid = _small_input(11)
    torch.manual_seed(5)
    net = P.VoxelResBackBone8x(PU.Cfg(), 5, np.asarray(grid)).to(DEV).train()
    sync = torch.nn.SyncBatchNorm.convert_sync_batchnorm(P.VoxelResBackBone8x(PU.Cfg(), 5, np.asarray(grid))).to(DEV).train()
    sync.load_state_dict(net.state_dict())
    n_sync = sum(isinstance(m, torch.nn.SyncBatchNorm) for m in sync.modules())
    assert n_sync == sum(isinstance(m, torch.nn.BatchNorm1d) for m in net.modules()) > 0
    calls = []
    real = dist.all_reduce
    dist.init_process_group("gloo", init_method=f"file://{tmp_path / 'pg'}", rank=0, world_size=1)
    try:
        dist.all_reduce = lambda *a, **k: (calls.append(1), real(*a, **k))[1]
        ref = _backbone_step(net, vf, coords, prec, 1)
        got = _backbone_step(sync, vf, coords, prec, 1)
        assert not calls
        sync.eval()
        with torch.no_grad():
            sync({"voxel_features": vf, "voxel_coords": coords, "batch_size": 2})
        assert not calls
    finally:
        dist.all_reduce = real
        dist.destroy_process_group()
    for u, v in zip(ref, got):
        assert torch.equal(u, v)
    sd_n, sd_s = net.state_dict(), sync.state_dict()
    assert list(sd_n) == list(sd_s)
    for k in sd_n:
        assert torch.equal(sd_n[k], sd_s[k]), k
    for (k, p), (_, q) in zip(net.named_parameters(), sync.named_parameters()):
        assert torch.equal(p.grad, q.grad), k


def test_momentum_none_is_refused():
    ops = _ops()
    bn = torch.nn.SyncBatchNorm(16, momentum=None).to(DEV).train()
    with pytest.raises(NotImplementedError, match="momentum=None"):
        ops.sync_group(bn)


# ---------------------------------------------------------------------------------------------- 3. two processes
def _two_rank_input(seed, empty_rank=None):
    """Two frames of different sizes (rank r runs frame r); empty_rank: that frame has no voxels."""
    sizes = [5200, 3700]
    if empty_rank is not None:
        sizes[empty_rank] = 0
    shape = [41, 200, 176]
    coords = _random_frames(sizes, shape, seed)
    vf = torch.randn((coords.shape[0], 5), generator=torch.Generator().manual_seed(seed))
    return vf, torch.from_numpy(coords), [176, 200, 40], sizes


def _worker(rank, world, backend, init, case, prec, out_dir):
    import toda_b200.pcdet_plugin as P
    from toda_b200 import dist as TD
    from toda_b200.spconv_compat import pytorch as G
    torch.cuda.set_device(rank)
    dist.init_process_group(backend, init_method=f"file://{init}", rank=rank, world_size=world,
                            timeout=datetime.timedelta(seconds=120))
    try:
        calls = []
        real = dist.all_reduce

        def counting(*a, **k):
            calls.append(1)
            return real(*a, **k)
        dist.all_reduce = counting
        vf, coords, grid, _ = _two_rank_input(21, 1 if case == "empty_rank" else None)
        sel = coords[:, 0] == rank
        c = coords[sel].clone()
        c[:, 0] = 0
        v = vf[sel].to(DEV).requires_grad_(True)
        c = c.to(DEV)
        torch.manual_seed(5)
        if case == "shim":
            net = _shim_net()
        else:
            net = P.VoxelResBackBone8x(PU.Cfg(), 5, np.asarray(grid))
        net = torch.nn.SyncBatchNorm.convert_sync_batchnorm(net).to(DEV)
        net.train(case != "eval")
        G.set_conv_precision(prec)
        if case == "shim":
            out = net(G.SparseConvTensor(v, c, [41, 200, 176], 1)).dense()
        else:
            hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
            out = hc(net({"voxel_features": v, "voxel_coords": c, "batch_size": 1}))["spatial_features"]
        res = {"out": out.detach().cpu()}
        if case != "eval":
            cot = torch.randn((2,) + tuple(out.shape[1:]), generator=torch.Generator().manual_seed(100))[rank].to(DEV)
            bucket = TD.FlatGradBucket(net.parameters()) if backend == "nccl" else None
            if bucket is not None:
                bucket.zero()
            (out * cot).sum().backward()
            if bucket is not None:
                bucket.all_reduce_mean()
            torch.cuda.synchronize()
            res["dv"] = v.grad.detach().cpu()
            res["grads"] = {k: p.grad.detach().cpu() for k, p in net.named_parameters()}
        res["state"] = {k: t.detach().cpu() for k, t in net.state_dict().items()}
        res["calls"] = len(calls)
        dist.all_reduce = real
        torch.save(res, os.path.join(out_dir, f"{rank}.pt"))
    finally:
        dist.destroy_process_group()


def _shim_net():
    """pcdet's post_act_block chain as plain SparseSequential modules (conv, BatchNorm1d, ReLU)."""
    from toda_b200.spconv_compat import pytorch as G
    nn = torch.nn
    return G.SparseSequential(
        G.SubMConv3d(5, 16, 3, padding=1, bias=False, indice_key="s1"), nn.BatchNorm1d(16, eps=1e-3, momentum=0.01), nn.ReLU(),
        G.SparseConv3d(16, 32, 3, stride=2, padding=1, bias=False, indice_key="d2"), nn.BatchNorm1d(32, eps=1e-3, momentum=0.01),
        nn.ReLU(),
        G.SubMConv3d(32, 32, 3, padding=1, bias=False, indice_key="s2"), nn.BatchNorm1d(32, eps=1e-3, momentum=0.01), nn.ReLU())


def _union_reference(case, prec):
    import toda_b200.pcdet_plugin as P
    from toda_b200.spconv_compat import pytorch as G
    vf, coords, grid, sizes = _two_rank_input(21, 1 if case == "empty_rank" else None)
    torch.manual_seed(5)
    net = (_shim_net() if case == "shim" else P.VoxelResBackBone8x(PU.Cfg(), 5, np.asarray(grid))).to(DEV)
    net.train(case != "eval")
    v = vf.to(DEV).requires_grad_(True)
    c = coords.to(DEV)
    G.set_conv_precision(prec)
    try:
        if case == "shim":
            out = net(G.SparseConvTensor(v, c, [41, 200, 176], 2)).dense()
        else:
            hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
            out = hc(net({"voxel_features": v, "voxel_coords": c, "batch_size": 2}))["spatial_features"]
        res = {"out": out.detach().cpu()}
        if case != "eval":
            cot = torch.randn((2,) + tuple(out.shape[1:]), generator=torch.Generator().manual_seed(100)).to(DEV)
            (out * cot).sum().backward()
            res["dv"] = v.grad.detach().cpu()
            res["grads"] = {k: p.grad.detach().cpu() for k, p in net.named_parameters()}
    finally:
        G.set_conv_precision("fp32")
    res["state"] = {k: t.detach().cpu() for k, t in net.state_dict().items()}
    res["sizes"] = sizes
    return res


def _rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def _compare(ranks, ref, prec, case, averaged):
    bound = 2e-2 if prec == "bf16" else None

    def close(got, want, what):
        if bound is None:
            PU.assert_close(got.double().numpy(), want.double().numpy(), rtol=1e-4, atol_scale=1e-5, what=what)
        else:
            e = _rel_l2(got, want)
            print(f"{what}: rel-L2 {e:.3e}")
            assert e <= bound, (what, e)
    sizes = ref["sizes"]
    offs = np.cumsum([0] + sizes)
    for r, res in enumerate(ranks):
        close(res["out"][0], ref["out"][r], f"{case} rank {r} output")
        if "dv" in res:
            close(res["dv"], ref["dv"][offs[r]:offs[r + 1]], f"{case} rank {r} d voxel_features")
    for k, t in ref["state"].items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            assert torch.equal(ranks[0]["state"][k], ranks[1]["state"][k]), k
            close(ranks[0]["state"][k], t, f"{case} {k}")
        elif k.endswith("num_batches_tracked"):
            assert int(ranks[0]["state"][k]) == int(ranks[1]["state"][k]) == int(t), k
    if "grads" in ref:
        for k, want in ref["grads"].items():
            got = ranks[0]["grads"][k] if averaged else (ranks[0]["grads"][k] + ranks[1]["grads"][k]) / 2
            if averaged:
                assert torch.equal(ranks[0]["grads"][k], ranks[1]["grads"][k]), k
            close(got, want / 2, f"{case} averaged grad {k}")


def _spawn(backend, case, prec):
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as d:
        init = os.path.join(d, "pg")
        mp.spawn(_worker, args=(2, backend, init, case, prec, d), nprocs=2, join=True)
        return [torch.load(os.path.join(d, f"{r}.pt")) for r in range(2)]


two_gpus = pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs 2 GPUs")


@two_gpus
@pytest.mark.parametrize("case,prec", [("unequal", "fp32"), ("unequal", "bf16"), ("empty_rank", "fp32"), ("shim", "fp32"),
                                       ("eval", "fp32")])
def test_two_processes_gloo_vs_union(case, prec):
    """gloo over CUDA tensors: a missing collective fails with the process group's timeout instead of hanging."""
    ranks = _spawn("gloo", case, prec)
    ref = _union_reference(case, prec)
    _compare(ranks, ref, prec, case, averaged=False)
    n_bn = sum(1 for k in ref["state"] if k.endswith("running_mean"))
    for res in ranks:
        assert res["calls"] == (0 if case == "eval" else 2 * n_bn), res["calls"]


@two_gpus
def test_two_processes_nccl_flat_grad_bucket():
    """The production path: NCCL, the collectives on the current stream, and FlatGradBucket averaging the gradients."""
    ranks = _spawn("nccl", "unequal", "fp32")
    ref = _union_reference("unequal", "fp32")
    _compare(ranks, ref, "fp32", "nccl", averaged=True)
