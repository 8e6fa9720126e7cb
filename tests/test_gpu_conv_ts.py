"""Row-cache / TMEM-operand convolution kernel (csrc/conv_ts.cu, toda_spconv_fwd with a tile plan) against the round-1 tensor-core
kernels on the same tables: same bf16 operands, same K order, fp32 accumulation in TMEM => bit-identical outputs and
BatchNorm sums.  Covers every conv geometry of VoxelResBackBone8x (SubM, stride-2 forward, parity-sorted dgrad with
out_rows, the (3,1,1) conv_out), the 4/5-channel input layer, ragged tails and plans that overflow the slab
(global-memory fallback rows)."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _both(x, cin, nbr, n_out, kvol, w, cout, plan, masks, out_rows=None, bias=None):
    from toda_b200 import ops
    xb = x.to(torch.bfloat16) if cin >= 16 else None
    outs = []
    for pl in (None, plan):
        sums = torch.zeros(2 * cout, dtype=torch.float64, device=x.device)
        y = ops._conv_call(x, xb, cin, nbr, n_out, kvol, w, cout, bias, ops.CONV_BF16, tile_masks=masks, plan=pl, bn_sums=sums,
                           out_rows=out_rows)
        torch.cuda.synchronize()
        outs.append((y, sums))
    return outs


@pytest.mark.parametrize("n,cin,cout", [(1, 16, 16), (127, 32, 32), (129, 64, 64), (5000, 128, 128), (20000, 5, 16), (40000, 16, 32),
                                        (30000, 64, 32), (30000, 128, 64)])
def test_plan_kernel_matches_round1_kernel_subm(n, cin, cout):
    from toda_b200 import ops
    shape, batch = [11, 200, 200], 2
    feats, idx = PU.random_sparse(n + cin, batch, shape, n, cin)
    index = ops.OccupancyIndex(batch, shape, torch.device(DEV, 0), "ts")
    index.insert(torch.from_numpy(idx).to(DEV))
    index.build(n)
    prev = ops.tile_plans_enabled()
    ops.set_tile_plans(True)
    try:
        rb = ops.rulebook_subm(index, [3, 3, 3], channels=max(cin, cout))
    finally:
        ops.set_tile_plans(prev)
    assert rb.plan is not None
    x = torch.from_numpy(feats).to(DEV)
    w = torch.randn(27, cin, cout, device=DEV) * 0.1
    bias = torch.randn(cout, device=DEV)
    (ya, sa), (yb, sb) = _both(x, cin, rb.nbr_fwd, rb.n_out, 27, w, cout, rb.plan, rb.tile_masks, bias=bias)
    index.release()
    assert torch.equal(ya, yb)
    assert torch.equal(sa, sb) or float((sa - sb).abs().max() / sa.abs().max()) < 1e-12


def test_plan_kernel_full_size_chain_all_geometries():
    """4 full-size nuScenes-shaped frames: SubM at every level, every strided conv forward and (parity-sorted) dgrad."""
    from toda_b200 import ops, synth
    cfg = synth.CONFIGS["nus_0075"]
    frames, collated = synth.make_batch("nus_0075", 4)
    dev = torch.device(DEV, 0)
    offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(dev)
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    _, coords, _, _ = ops.voxelize(torch.from_numpy(collated).to(dev), offs, cfg["pc_range"], cfg["voxel_size"], 10, 120000,
                                   xyz_col=1, feat_col=1, num_features=5, order=ops.ORDER_CANONICAL, grid=grid)
    shape = [int(grid[2]) + 1, int(grid[1]), int(grid[0])]
    index = ops.OccupancyIndex(4, shape, dev, "tsfull")
    index.insert(coords)
    index.build(coords.shape[0], known_n=coords.shape[0])
    chain = [(16, 32, [3, 3, 3], [2, 2, 2], [1, 1, 1]), (32, 64, [3, 3, 3], [2, 2, 2], [1, 1, 1]),
             (64, 128, [3, 3, 3], [2, 2, 2], [0, 1, 1]), (128, 128, [3, 1, 1], [2, 1, 1], [0, 0, 0])]
    torch.manual_seed(0)
    ops.set_tile_plans(True)
    try:
        for cin, cout, k, s, p in chain:
            rbs = ops.rulebook_subm(index, [3, 3, 3], channels=cin)
            x = torch.randn(rbs.n_in, cin, device=dev)
            w = torch.randn(27, cin, cin, device=dev) * 0.1
            (ya, sa), (yb, sb) = _both(x, cin, rbs.nbr_fwd, rbs.n_out, 27, w, cin, rbs.plan, rbs.tile_masks)
            assert torch.equal(ya, yb) and torch.equal(sa, sb), ("subm", cin)
            rb, index = ops.rulebook_sparse(index, k, s, p, ("tsfull", cin), cin=cin, cout=cout)
            kvol = k[0] * k[1] * k[2]
            w = torch.randn(kvol, cin, cout, device=dev) * 0.1
            (ya, sa), (yb, sb) = _both(x, cin, rb.nbr_fwd, rb.n_out, kvol, w, cout, rb.plan, rb.tile_masks)
            assert torch.equal(ya, yb) and torch.equal(sa, sb), ("down fwd", cin, cout)
            dy = torch.randn(rb.n_out, cout, device=dev)
            wt = torch.randn(kvol, cout, cin, device=dev) * 0.1
            if rb.dgrad_order is not None:
                (ya, _), (yb, _) = _both(dy, cout, rb.nbr_bwd_sorted, rb.n_in, kvol, wt, cin, rb.dgrad_plan, rb.dgrad_tile_masks,
                                         out_rows=rb.dgrad_order)
            else:
                (ya, _), (yb, _) = _both(dy, cout, rb.nbr_bwd, rb.n_in, kvol, wt, cin, rb.dgrad_plan, None)
            assert torch.equal(ya, yb), ("down dgrad", cin, cout)
    finally:
        ops.set_tile_plans(False)


def test_backbone_step_with_plans_is_bit_identical():
    """VoxelResBackBone8x fwd+bwd (bf16 mode, train-mode BN) with and without tile plans: identical outputs and gradients."""
    import toda_b200.pcdet_plugin as P
    from toda_b200 import ops
    from toda_b200.spconv_compat import pytorch as G
    g = PU.load_golden("backbone_res.npz")
    hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
    vf = torch.from_numpy(g["voxel_features"]).to(DEV)
    vc = torch.from_numpy(g["voxel_coords"]).float().to(DEV)
    cot = torch.randn(tuple(g["bev_shape"]), generator=torch.Generator().manual_seed(int(g["seed"])))
    res = []
    G.set_conv_precision("bf16")
    try:
        for plans in (False, True):
            ops.set_tile_plans(plans)
            _, net = PU.build_pair("VoxelResBackBone8x", 5, g["grid_size"], seed=int(g["seed"]))
            res.append(PU.run_backbone(net, hc, vf, vc, 2, cot=cot, train=True))
    finally:
        ops.set_tile_plans(False)
        G.set_conv_precision("fp32")
    a, b = res
    assert np.array_equal(a["spatial_features"], b["spatial_features"])
    assert np.array_equal(a["dvoxel_features"], b["dvoxel_features"])
    for k in a["grads"]:
        # (BatchNorm sums are fp64 atomics in both paths: order-dependent in the last bits)
        np.testing.assert_allclose(a["grads"][k], b["grads"][k], rtol=1e-5, atol=1e-7, err_msg=k)


def test_strided_forward_stress_on_second_rank_frames():
    """Regression guard for a deadlock of the row-cache kernel that showed only on the frames the SECOND rank of a
    multi-GPU run gets (synthetic frames 12-15), and only a few times in ten 20-step runs: on the 32->64 stride-2 forward
    conv the second slab-loader warp waited on slab_empty by itself, fell two uses of a buffer behind in units where it had
    no block to fetch, and its parity wait never passed again.  (It now follows the first loader through a named
    barrier.)  The test repeats that layer 400 times on those frames and checks every launch against the first.  (The
    kernel stays opt-in: a second, rarer hang of the same family was still open at the end of round 2, see ops.py.)"""
    from toda_b200 import ops, synth
    cfg = synth.CONFIGS["nus_0075"]
    frames, collated = synth.make_batch("nus_0075", 4, first_frame=12)
    dev = torch.device(DEV, 0)
    offs = torch.from_numpy(np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)).to(dev)
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    _, coords, _, _ = ops.voxelize(torch.from_numpy(collated).to(dev), offs, cfg["pc_range"], cfg["voxel_size"], 10, 120000, xyz_col=1,
                                   feat_col=1, num_features=5, order=ops.ORDER_CANONICAL, grid=grid)
    shape = [int(grid[2]) + 1, int(grid[1]), int(grid[0])]
    index = ops.OccupancyIndex(4, shape, dev, "stress")
    index.insert(coords)
    index.build(coords.shape[0], known_n=coords.shape[0])
    ops.set_tile_plans(True)
    try:
        _, index = ops.rulebook_sparse(index, [3, 3, 3], [2, 2, 2], [1, 1, 1], ("stress", 1), cin=16, cout=32)
        rb, index3 = ops.rulebook_sparse(index, [3, 3, 3], [2, 2, 2], [1, 1, 1], ("stress", 2), cin=32, cout=64)
    finally:
        ops.set_tile_plans(False)
    assert rb.plan is not None
    x = torch.randn(rb.n_in, 32, device=dev)
    xb = x.to(torch.bfloat16)
    w = torch.randn(27, 32, 64, device=dev) * 0.1
    ref = None
    for i in range(400):
        y = ops._conv_call(x, xb, 32, rb.nbr_fwd, rb.n_out, 27, w, 64, None, ops.CONV_BF16, tile_masks=rb.tile_masks, plan=rb.plan)
        if i % 50 == 0:
            torch.cuda.synchronize()
            if ref is None:
                ref = y.clone()
            assert torch.equal(y, ref)
    torch.cuda.synchronize()
    index3.release()
