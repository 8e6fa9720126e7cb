"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle and the committed golden
fixtures.  Integers (coords, counts, membership, rulebook pairs) bit-exact; fp32 within rtol 1e-4."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _lib_loaded():
    from toda_b200 import _C
    lib = _C.lib()
    sm, major, minor = [__import__("ctypes").c_int() for _ in range(3)]
    _C.check(lib.toda_device_info(sm, major, minor), "toda_device_info")
    assert major.value >= 10, f"needs sm_100 (got {major.value}.{minor.value})"


# ------------------------------------------------------------------------------------------ K1 / K2
@pytest.mark.parametrize("case", ["crop_nus", "crop_nus_capped", "crop_waymo", "coarse_full_nus"])
def test_voxelize_golden(case):
    from toda_b200 import ops
    c = PU.golden_cases(PU.load_golden("voxelize.npz"))[case]
    pts, k, mv = c["points"], int(c["max_points"]), int(c["max_voxels"])
    want = (c["voxels"], np.pad(c["voxel_coords"], ((0, 0), (1, 0))).astype(np.int32), c["voxel_num_points"],
            np.array([c["voxels"].shape[0]] * 2))
    got = PU.gpu_voxelize_batch([pts], c["pc_range"], c["voxel_size"], k, mv, ops.ORDER_FIRST_APPEARANCE)
    PU.assert_voxels_equal(got, want, exact_order=True)          # same rows in the same order as the reference
    got = PU.gpu_voxelize_batch([pts], c["pc_range"], c["voxel_size"], k, mv, ops.ORDER_CANONICAL)
    PU.assert_voxels_equal(got, want, exact_order=False)
    o = PU.canonical_order(got[1])
    assert np.array_equal(o, np.arange(len(o)))                  # canonical mode really is (b,z,y,x)-sorted
    vf = ops.mean_vfe(torch.from_numpy(c["voxels"]).to(DEV), torch.from_numpy(c["voxel_num_points"]).to(DEV))
    PU.assert_close(vf.cpu().numpy(), c["voxel_features"], what="voxel_features")
    vf2 = ops.mean_vfe(torch.from_numpy(c["voxels"]).to(DEV), torch.from_numpy(c["voxel_num_points"]).float().to(DEV))
    assert torch.equal(vf, vf2)                                  # float counts (load_data_to_gpu) == int counts


def test_voxelize_ragged_batch_with_empty_frame_and_caps():
    from toda_b200 import ops
    rng = np.random.default_rng(5)
    pcr, vs = [-8.0, -8.0, -1.5, 8.0, 8.0, 1.5], [0.5, 0.5, 0.25]

    def frame(n):
        p = rng.random((n, 4), dtype=np.float32)
        p[:, :3] = p[:, :3] * np.array([20, 20, 4], np.float32) - np.array([10, 10, 2], np.float32)
        return p
    frames = [frame(5000), np.zeros((0, 4), np.float32), frame(1), frame(20000), frame(777)]
    frames[3][:4000, :3] = frames[3][0, :3]           # 4000 duplicates of one point: a crowded voxel
    frames[4][5] = [8.0, 0, 0, 1]                      # x == hi -> dropped
    frames[4][6] = [np.nan, 0, 0, 1]
    for k, mv in [(3, 300), (1, 100000), (10, 50)]:
        want = PU.oracle_voxelize_batch(frames, pcr, vs, k, mv)
        got = PU.gpu_voxelize_batch(frames, pcr, vs, k, mv, ops.ORDER_FIRST_APPEARANCE)
        PU.assert_voxels_equal(got, want, exact_order=True)
        got = PU.gpu_voxelize_batch(frames, pcr, vs, k, mv, ops.ORDER_CANONICAL)
        PU.assert_voxels_equal(got, want, exact_order=False)


def test_voxelize_all_empty():
    from toda_b200 import ops
    got = PU.gpu_voxelize_batch([np.zeros((0, 5), np.float32)] * 2, [-8, -8, -1, 8, 8, 1], [0.5, 0.5, 0.5], 3, 10,
                                ops.ORDER_FIRST_APPEARANCE)
    assert got[0].shape == (0, 3, 5) and got[3].tolist() == [0, 0, 0]


@pytest.mark.parametrize("cfg_name,train", [("nus_0075", True), ("waymo_010", True), ("nus_010", False)])
def test_voxelize_full_size_frames(cfg_name, train):
    """BASELINE.json configs at their real grid sizes, batch of 2, collated `points` layout [b,x,y,z,...]."""
    from toda_b200 import ops, synth
    cfg = synth.CONFIGS[cfg_name]
    frames, collated = synth.make_batch(cfg_name, 2)
    mv = cfg["max_voxels"]["train" if train else "test"]
    want = PU.oracle_voxelize_batch(frames, cfg["pc_range"], cfg["voxel_size"], cfg["max_points"], mv)
    offs = torch.tensor(np.cumsum([0] + [f.shape[0] for f in frames]), dtype=torch.int32, device=DEV)
    pts = torch.from_numpy(collated).to(DEV)
    for order in (ops.ORDER_FIRST_APPEARANCE, ops.ORDER_CANONICAL):
        v, c, n, counts = ops.voxelize(pts, offs, cfg["pc_range"], cfg["voxel_size"], cfg["max_points"], mv,
                                       num_features=cfg["num_features"], xyz_col=1, feat_col=1, order=order)
        got = (v.cpu().numpy(), c.cpu().numpy(), n.cpu().numpy(), counts.cpu().numpy())
        PU.assert_voxels_equal(got, want, exact_order=(order == ops.ORDER_FIRST_APPEARANCE))
    # size-independent properties: every kept point is inside its voxel; counts add up; idempotence
    assert int(n.sum()) <= collated.shape[0] and (n >= 1).all() and (n <= cfg["max_points"]).all()
    v2, c2, n2, _ = ops.voxelize(pts, offs, cfg["pc_range"], cfg["voxel_size"], cfg["max_points"], mv,
                                 num_features=cfg["num_features"], xyz_col=1, feat_col=1, order=ops.ORDER_CANONICAL)
    assert torch.equal(v, v2) and torch.equal(c, c2) and torch.equal(n, n2)       # deterministic run to run


def test_mean_vfe_backward_matches_autograd():
    from toda_b200 import ops
    rng = np.random.default_rng(0)
    v = torch.from_numpy(rng.standard_normal((1000, 7, 5)).astype(np.float32))
    n = torch.from_numpy(rng.integers(0, 8, 1000).astype(np.int32))
    g = torch.from_numpy(rng.standard_normal((1000, 5)).astype(np.float32))
    v1 = v.clone().requires_grad_(True)
    ref = v1.sum(dim=1) / torch.clamp_min(n.float().view(-1, 1), 1.0)
    ref.backward(g)
    v2 = v.clone().to(DEV).requires_grad_(True)
    out = ops.mean_vfe(v2, n.to(DEV))
    out.backward(g.to(DEV))
    PU.assert_close(out.detach().cpu().numpy(), ref.detach().numpy(), what="mean fwd")
    PU.assert_close(v2.grad.cpu().numpy(), v1.grad.numpy(), what="mean bwd")


# ------------------------------------------------------------------------------------------ K3 / K4
@pytest.mark.parametrize("shape,n", [([7, 9, 11], 300), ([41, 64, 64], 5000), ([5, 33, 70], 2000)])
def test_subm_rulebook_bit_exact(shape, n):
    from oracle import spconv_oracle as S
    from toda_b200 import ops
    feats, idx = PU.random_sparse(1, 3, shape, n, 4)
    shuffled = idx[np.random.default_rng(2).permutation(n)]
    index = ops.OccupancyIndex(3, shape, torch.device(DEV, 0), "t")
    index.insert(torch.from_numpy(shuffled).to(DEV))
    coords = index.build(n)
    assert np.array_equal(coords.cpu().numpy(), idx)               # canonical order out of any input order
    rows = index.rows(torch.from_numpy(shuffled).to(DEV)).cpu().numpy()
    assert np.array_equal(idx[rows], shuffled)
    rb = ops.rulebook_subm(index, [3, 3, 3])
    got = PU.table_to_canonical_pairs(rb.nbr_fwd.cpu().numpy(), idx, idx, shape, shape)
    want = S.rulebook_pairs_canonical(idx, idx, S.subm_rulebook(idx, shape, [3, 3, 3]), shape, shape)
    assert np.array_equal(got, want)
    # release leaves the shared buffer clean: a different coordinate set built next sees no stale marks
    index.release()
    _, idx2 = PU.random_sparse(8, 3, shape, n // 2, 4)
    index2 = ops.OccupancyIndex(3, shape, torch.device(DEV, 0), "t")
    index2.insert(torch.from_numpy(idx2).to(DEV))
    assert np.array_equal(index2.build(n).cpu().numpy(), idx2)
    index2.release()


@pytest.mark.parametrize("k,s,p", [((3, 3, 3), (2, 2, 2), (1, 1, 1)), ((3, 3, 3), (2, 2, 2), (0, 1, 1)),
                                   ((3, 1, 1), (2, 1, 1), (0, 0, 0)), ((3, 3, 3), (1, 1, 1), (0, 0, 0))])
def test_sparse_rulebook_bit_exact(k, s, p):
    from oracle import spconv_oracle as S
    from toda_b200 import ops
    shape, n = [11, 30, 37], 3000
    feats, idx = PU.random_sparse(3, 2, shape, n, 4)
    index = ops.OccupancyIndex(2, shape, torch.device(DEV, 0), "t")
    index.insert(torch.from_numpy(idx).to(DEV))
    index.build(n)
    rb, index_out = ops.rulebook_sparse(index, list(k), list(s), list(p), "t_out")
    oi, oshape, pairs = S.sparse_rulebook(idx, shape, list(k), list(s), list(p))
    assert rb.out_shape == oshape
    assert np.array_equal(rb.out_coords.cpu().numpy(), oi)          # output coords, canonical order, bit-exact
    want = S.rulebook_pairs_canonical(idx, oi, pairs, shape, oshape)
    got = PU.table_to_canonical_pairs(rb.nbr_fwd.cpu().numpy(), idx, oi, shape, oshape)
    assert np.array_equal(got, want)
    # the input-stationary table holds the same pairs, transposed
    tb = rb.nbr_bwd.cpu().numpy()
    rows = []
    for kk in range(tb.shape[0]):
        i = np.nonzero(tb[kk] >= 0)[0]
        rows.append((i.astype(np.int64), tb[kk][i].astype(np.int64)))
    got_b = S.rulebook_pairs_canonical(idx, oi, rows, shape, oshape)
    assert np.array_equal(got_b, want)


# ------------------------------------------------------------------------------------------ K5-K7
def _conv_pair(subm, cin, cout, bias, k, s, p):
    from oracle import spconv_oracle as S
    from toda_b200.spconv_compat import pytorch as G
    torch.manual_seed(0)
    if subm:
        a = S.SubMConv3d(cin, cout, k, padding=p, bias=bias, indice_key="a")
        b = G.SubMConv3d(cin, cout, k, padding=p, bias=bias, indice_key="a")
    else:
        a = S.SparseConv3d(cin, cout, k, stride=s, padding=p, bias=bias, indice_key="a")
        b = G.SparseConv3d(cin, cout, k, stride=s, padding=p, bias=bias, indice_key="a")
    b.load_state_dict(a.state_dict())
    return a, b.to(DEV), S, G


@pytest.mark.parametrize("subm,cin,cout,bias,k,s,p", [
    (True, 5, 16, False, 3, 1, 1), (True, 4, 16, False, 3, 1, 1), (True, 16, 16, True, 3, 1, 1),
    (True, 32, 32, True, 3, 1, 1), (True, 64, 64, True, 3, 1, 1), (True, 128, 128, True, 3, 1, 1),
    (False, 16, 32, False, 3, 2, 1), (False, 32, 64, False, 3, 2, 1), (False, 64, 128, False, 3, 2, (0, 1, 1)),
    (False, 128, 128, False, (3, 1, 1), (2, 1, 1), 0), (False, 64, 64, False, 3, 2, (0, 1, 1))])
def test_conv_fwd_bwd_vs_oracle(subm, cin, cout, bias, k, s, p):
    a, b, S, G = _conv_pair(subm, cin, cout, bias, k, s, p)
    shape, n, batch = [9, 24, 31], 2500, 2
    feats, idx = PU.random_sparse(7, batch, shape, n, cin)
    perm = np.random.default_rng(1).permutation(n)                  # feed the GPU path a shuffled row order
    fa = torch.from_numpy(feats).requires_grad_(True)
    fb = torch.from_numpy(feats[perm]).to(DEV).requires_grad_(True)
    ya = a(S.SparseConvTensor(fa, torch.from_numpy(idx), shape, batch))
    yb = b(G.SparseConvTensor(fb, torch.from_numpy(idx[perm]).to(DEV), shape, batch))
    assert yb.spatial_shape == ya.spatial_shape
    assert np.array_equal(yb.indices.cpu().numpy(), ya.indices.numpy())   # both canonical
    PU.assert_close(yb.features.detach().cpu().numpy(), ya.features.detach().numpy(), what="conv fwd")
    g = torch.randn(ya.features.shape, generator=torch.Generator().manual_seed(3))
    ya.features.backward(g)
    yb.features.backward(g.to(DEV))
    PU.assert_close(fb.grad.cpu().numpy(), fa.grad.numpy()[perm], what="dgrad")
    PU.assert_close(b.weight.grad.cpu().numpy(), a.weight.grad.numpy(), what="wgrad")
    if bias:
        PU.assert_close(b.bias.grad.cpu().numpy(), a.bias.grad.numpy(), what="bias grad")


def test_conv_empty_and_tiny_inputs():
    a, b, S, G = _conv_pair(True, 16, 16, True, 3, 1, 1)
    for n in (0, 1, 3):
        feats, idx = PU.random_sparse(9, 1, [5, 6, 7], n, 16)
        yb = b(G.SparseConvTensor(torch.from_numpy(feats).to(DEV), torch.from_numpy(idx).to(DEV), [5, 6, 7], 1))
        ya = a(S.SparseConvTensor(torch.from_numpy(feats), torch.from_numpy(idx), [5, 6, 7], 1))
        assert yb.features.shape == ya.features.shape
        if n:
            PU.assert_close(yb.features.detach().cpu().numpy(), ya.features.detach().numpy(), what="tiny conv")


# ------------------------------------------------------------------------------------------ K8 / K9
@pytest.mark.parametrize("c,n,res,relu,train", [(16, 5000, False, True, True), (128, 3001, True, True, True),
                                                (64, 1, False, True, True), (32, 4000, True, False, True),
                                                (16, 2000, False, True, False), (5, 777, True, True, True),
                                                (32, 0, True, True, True)])
def test_bn_act_vs_torch(c, n, res, relu, train):
    from toda_b200 import ops
    torch.manual_seed(1)
    bn_a = torch.nn.BatchNorm1d(c, eps=1e-3, momentum=0.01)
    with torch.no_grad():
        bn_a.weight.uniform_(0.5, 1.5)
        bn_a.bias.uniform_(-0.5, 0.5)
        bn_a.running_mean.uniform_(-0.2, 0.2)
        bn_a.running_var.uniform_(0.5, 2.0)
    bn_b = torch.nn.BatchNorm1d(c, eps=1e-3, momentum=0.01)
    bn_b.load_state_dict(bn_a.state_dict())
    bn_b = bn_b.to(DEV)
    bn_a.train(train)
    bn_b.train(train)
    if n == 1 and train:
        bn_a.eval()       # torch refuses batch statistics over one row; compare the n>1 contract only
        bn_b.eval()
    y = torch.randn(n, c) * 2 + 0.3
    r = torch.randn(n, c) if res else None
    g = torch.randn(n, c)
    ya = y.clone().requires_grad_(True)
    ra = r.clone().requires_grad_(True) if res else None
    oa = PU.bn_act_torch(ya, bn_a, ra, relu)
    oa.backward(g)
    yb = y.clone().to(DEV).requires_grad_(True)
    rb = r.clone().to(DEV).requires_grad_(True) if res else None
    ob = ops.bn_act(yb, bn_b, rb, relu)
    ob.backward(g.to(DEV))
    PU.assert_close(ob.detach().cpu().numpy(), oa.detach().numpy(), what="bn fwd")
    PU.assert_close(yb.grad.cpu().numpy(), ya.grad.numpy(), rtol=1e-3, what="bn dy")
    PU.assert_close(bn_b.weight.grad.cpu().numpy(), bn_a.weight.grad.numpy(), rtol=1e-3, what="dgamma")
    PU.assert_close(bn_b.bias.grad.cpu().numpy(), bn_a.bias.grad.numpy(), rtol=1e-3, what="dbeta")
    if res:
        PU.assert_close(rb.grad.cpu().numpy(), ra.grad.numpy(), what="dresidual")
    PU.assert_close(bn_b.running_mean.cpu().numpy(), bn_a.running_mean.numpy(), what="running_mean")
    PU.assert_close(bn_b.running_var.cpu().numpy(), bn_a.running_var.numpy(), what="running_var")
    # (n = 0: empty output, zero parameter gradients, running statistics unchanged, the batch still counted -- as torch)
    assert int(bn_b.num_batches_tracked) == int(bn_a.num_batches_tracked)


def test_bev_scatter_bit_exact_and_backward():
    from oracle import spconv_oracle as S
    from toda_b200 import ops
    shape, n, c, batch = [2, 45, 52], 1500, 128, 3
    feats, idx = PU.random_sparse(4, batch, shape, n, c)
    dense = S.SparseConvTensor(torch.from_numpy(feats), torch.from_numpy(idx), shape, batch).dense()
    want = dense.view(batch, c * shape[0], shape[1], shape[2]).numpy()
    f = torch.from_numpy(feats).to(DEV).requires_grad_(True)
    got = ops.bev_scatter(f, torch.from_numpy(idx).to(DEV), batch, *shape)
    assert np.array_equal(got.detach().cpu().numpy().view(np.uint32), want.view(np.uint32))   # exact copy
    g = torch.randn(got.shape)
    got.backward(g.to(DEV))
    want_g = g.view(batch, c, *shape)[idx[:, 0], :, idx[:, 1], idx[:, 2], idx[:, 3]]
    assert torch.equal(f.grad.cpu(), want_g)


# ------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("cls,fname", [("VoxelResBackBone8x", "backbone_res.npz"), ("VoxelBackBone8x", "backbone_voxel.npz"),
                                       ("VoxelResBackBone8x", "backbone_res_stage2.npz")])
def test_backbone_vs_reference_golden(cls, fname):
    """Golden vectors produced through the reference's own spconv_backbone.py + height_compression.py.
    backbone_res_stage2: the TODA stage-2 geometry (z range -5..4.8 -> sparse_shape [50, ., .], F = 4, mixup / polar-swap
    samples; BASELINE configs[3])."""
    import toda_b200.pcdet_plugin as P
    g = PU.load_golden(fname)
    nf = int(g["voxel_features"].shape[1])
    if "stage2" in fname:
        assert int(g["grid_size"][2]) == 49
    twin, net = PU.build_pair(cls, nf, g["grid_size"], seed=int(g["seed"]))
    hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
    vf = torch.from_numpy(g["voxel_features"]).to(DEV)
    vc = torch.from_numpy(g["voxel_coords"]).float().to(DEV)       # float32 coords, as load_data_to_gpu delivers
    cot = torch.randn(tuple(g["bev_shape"]), generator=torch.Generator().manual_seed(int(g["seed"])))
    r = PU.run_backbone(net, hc, vf, vc, 2, cot=cot, train=True)
    f_sorted, i_sorted = PU.sort_rows(r["enc_features"], r["enc_indices"])
    assert np.array_equal(i_sorted, g["train_enc_indices"])
    PU.assert_close(f_sorted, g["train_enc_features"], what="encoded features")
    assert abs(r["loss"] - float(g["train_loss"])) < 1e-3 * max(1.0, abs(float(g["train_loss"])))
    names = [str(n) for n in g["grad_names"]]
    norms = np.array([np.linalg.norm(r["grads"][n].astype(np.float64)) for n in names])
    if "stage2" in fname:
        # This crop holds ONE activation (x_conv4, 2.3e-6 in the fp32 reference, 0 here) that sits on the ReLU kink: its mask
        # flips under fp32 accumulation-order noise and moves every gradient upstream of conv4 by ~0.5 % (verified element by
        # element with scripts/debug_stage2_golden.py: d x_conv4 agrees to 2e-6, conv_out's gradients to 2e-6, 1 flipped mask
        # of 120 320).  Gradients below the flip are therefore bounded in relative L2; everything else stays at rtol 1e-3.
        def rl2(a, b):
            a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
            return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
        assert rl2(r["dvoxel_features"], g["train_dvoxel_features"]) <= 2e-2
        np.testing.assert_allclose(norms, g["grad_norms"], rtol=2e-2, atol=1e-6 * float(g["grad_norms"].max()))
        assert rl2(r["grads"]["conv_input.0.weight"], g["grad_conv_input_weight"]) <= 2e-2
    else:
        # d loss / d voxel_features comes back in the caller's (golden) row order
        PU.assert_close(r["dvoxel_features"], g["train_dvoxel_features"], rtol=1e-3, what="d voxel_features")
        # conv biases feeding a BatchNorm have a mathematically zero gradient: their golden norms (~1e-3 next to
        # ~1e4 for the weights) are rounding noise, hence the absolute floor
        np.testing.assert_allclose(norms, g["grad_norms"], rtol=2e-3, atol=1e-6 * float(g["grad_norms"].max()))
        PU.assert_close(r["grads"]["conv_input.0.weight"], g["grad_conv_input_weight"], rtol=1e-3, atol_scale=1e-4, what="wgrad in")
    PU.assert_close(r["grads"]["conv_out.0.weight"], g["grad_conv_out_weight"], rtol=1e-3, atol_scale=1e-4, what="wgrad out")
    PU.assert_close(net.conv_input[1].running_mean.cpu().numpy(), g["running_mean_conv_input"], what="running_mean")
    PU.assert_close(net.conv_input[1].running_var.cpu().numpy(), g["running_var_conv_input"], what="running_var")
    for k in ["x_conv1", "x_conv2", "x_conv3", "x_conv4"]:
        fs, is_ = PU.sort_rows(r[k + "_features"], r[k + "_indices"])
        gs, gi = PU.sort_rows(g[f"train_{k}_features"], g[f"train_{k}_indices"])
        assert np.array_equal(is_, gi)
        PU.assert_close(fs, gs, what=k)
    # eval mode (running statistics) from a fresh copy of the initial weights
    twin2, net2 = PU.build_pair(cls, nf, g["grid_size"], seed=int(g["seed"]))
    with torch.no_grad():
        r2 = PU.run_backbone(net2, hc, vf, vc, 2, train=False)
    f2, i2 = PU.sort_rows(r2["enc_features"], r2["enc_indices"])
    assert np.array_equal(i2, g["eval_enc_indices"])
    PU.assert_close(f2, g["eval_enc_features"], what="eval encoded features")
    assert abs(float(r2["spatial_features"].astype(np.float64).sum()) - float(g["eval_bev_sum"])) < 1e-3 * abs(float(g["eval_bev_sum"])) + 1e-3


def test_smoke_entry():
    PU.run_smoke()


def test_compat_shim_runs_sequential_with_fused_bn():
    """spconv-shaped containers (what the reference's unmodified spconv_backbone.py builds) on the GPU shim."""
    from oracle import spconv_oracle as S
    from toda_b200.spconv_compat import pytorch as G
    torch.manual_seed(0)

    def build(sp):
        return sp.SparseSequential(sp.SubMConv3d(5, 16, 3, padding=1, bias=False, indice_key="s"),
                                   torch.nn.BatchNorm1d(16, eps=1e-3, momentum=0.01), torch.nn.ReLU(),
                                   sp.SparseConv3d(16, 32, 3, stride=2, padding=1, bias=False, indice_key="d"),
                                   torch.nn.BatchNorm1d(32, eps=1e-3, momentum=0.01), torch.nn.ReLU())
    a = build(S)
    b = build(G)
    b.load_state_dict(a.state_dict())
    b = b.to(DEV)
    feats, idx = PU.random_sparse(11, 2, [9, 20, 20], 1500, 5)
    ya = a(S.SparseConvTensor(torch.from_numpy(feats), torch.from_numpy(idx), [9, 20, 20], 2))
    yb = b(G.SparseConvTensor(torch.from_numpy(feats).to(DEV), torch.from_numpy(idx).to(DEV), [9, 20, 20], 2))
    assert np.array_equal(yb.indices.cpu().numpy(), ya.indices.numpy())
    PU.assert_close(yb.features.detach().cpu().numpy(), ya.features.detach().numpy(), what="sequential")
    PU.assert_close(yb.dense().detach().cpu().numpy(), ya.dense().detach().numpy(), what="dense")


@pytest.mark.parametrize("stride,padding,n", [((2, 2, 2), (1, 1, 1), 70001), ((2, 2, 2), (0, 1, 1), 1024), ((2, 1, 1), (0, 0, 0), 5000),
                                              ((1, 2, 1), (0, 1, 0), 33)])
def test_parity_order_is_a_stable_class_sort(stride, padding, n):
    """toda_parity_order == numpy stable argsort of the class code; the tile masks of the class-sorted table agree with it."""
    from toda_b200 import ops
    rng = np.random.default_rng(n)
    coords = np.stack([rng.integers(0, 3, n), rng.integers(0, 41, n), rng.integers(0, 300, n), rng.integers(0, 300, n)], 1).astype(np.int32)
    cls = np.zeros(n, np.int64)
    for a in range(3):
        cls = cls * stride[a] + (coords[:, 1 + a] + padding[a]) % stride[a]
    want = np.argsort(cls, kind="stable")
    c = torch.from_numpy(coords).cuda()
    table = torch.from_numpy(rng.integers(-1, 50, (27, n)).astype(np.int32) * (rng.random((27, n)) < 0.05) - (rng.random((27, n)) >= 0.5)).int().cuda()
    order, sorted_table = ops._dgrad_parity_order(c, table, list(stride), list(padding))
    assert np.array_equal(order.cpu().numpy(), want)
    assert torch.equal(sorted_table, table[:, order.long()])
    masks = ops.table_tile_masks(sorted_table).cpu().numpy().astype(np.uint32)
    t = sorted_table.cpu().numpy()
    for tile in range((n + 127) // 128):
        blk = t[:, tile * 128:(tile + 1) * 128]
        want_mask = sum((1 << k) for k in range(27) if (blk[k] >= 0).any())
        assert int(masks[tile]) == want_mask, tile


def test_two_shape_preserving_sparse_convs_without_indice_key():
    """SparseConv3d k3 s1 p1 keeps the spatial shape, and convs with indice_key=None share one tag: the output index must
    not alias (and un-mark) the input index (ADVICE r01: rulebook_sparse aliasing)."""
    from oracle import spconv_oracle as S
    from toda_b200.spconv_compat import pytorch as G
    torch.manual_seed(0)
    shape, n, batch = [9, 20, 20], 800, 2

    def build(sp):
        return sp.SparseSequential(sp.SparseConv3d(8, 8, 3, stride=1, padding=1, bias=True), sp.SparseConv3d(8, 16, 3, stride=1, padding=1, bias=False),
                                   sp.SparseConv3d(16, 8, 1, stride=1, padding=0, bias=False))
    a, b = build(S), build(G)
    b.load_state_dict(a.state_dict())
    b = b.to(DEV)
    feats, idx = PU.random_sparse(11, batch, shape, n, 8)
    fa = torch.from_numpy(feats).requires_grad_(True)
    fb = torch.from_numpy(feats).to(DEV).requires_grad_(True)
    ya = a(S.SparseConvTensor(fa, torch.from_numpy(idx), shape, batch))
    yb = b(G.SparseConvTensor(fb, torch.from_numpy(idx).to(DEV), shape, batch))
    fa_s, ia = PU.sort_rows(ya.features.detach().numpy(), ya.indices.numpy())
    fb_s, ib = PU.sort_rows(yb.features.detach().cpu().numpy(), yb.indices.cpu().numpy())
    assert np.array_equal(ia, ib)
    PU.assert_close(fb_s, fa_s, what="chained shape-preserving SparseConv3d")
    ya.features.sum().backward()
    yb.features.sum().backward()
    PU.assert_close(fb.grad.cpu().numpy(), fa.grad.numpy(), rtol=1e-3, what="dgrad through the chain")
