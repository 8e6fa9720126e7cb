"""Shared helpers for the parity tests and __graft_entry__.smoke(): run the CPU oracle and the CUDA path on the
same inputs and compare (bit-exact for integers, rtol 1e-4 for fp32)."""
import contextlib
import os

import numpy as np
import torch

from oracle import spconv_oracle as S
from oracle import voxelize as OV
from toda_b200.pcdet_plugin.backbones import make_backbones

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RTOL = 1e-4     # north-star tolerance for fp32 features / activations / gradients
# The backbone goldens were generated with 8 torch intra-op threads.  The oracle's fp32 results depend on the thread count
# (BatchNorm statistics and the GEMMs split their sums by thread), so a golden replays bit for bit only at that count.
GOLDEN_THREADS = 8


@contextlib.contextmanager
def golden_threads():
    prev = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(prev)


class Cfg(dict):
    __getattr__ = dict.get


def bn_act_torch(feat, bn, residual, relu):
    """What the fused K8 pass replaces, with stock torch ops (spconv_backbone.py L54-64)."""
    out = bn(feat)
    if residual is not None:
        out = out + residual
    return torch.relu(out) if relu else out


def bn_act_tensor_torch(x, bn, residual, relu):
    return x.replace_feature(bn_act_torch(x.features, bn, residual, relu))


def oracle_backbones():
    """The plugin's topology instantiated on the CPU oracle provider (same parameter names, order and init)."""
    return make_backbones(S, bn_act_tensor_torch)


def load_golden(name):
    return np.load(os.path.join(GOLDEN, name), allow_pickle=False)


def golden_cases(npz):
    cases = {}
    for key in npz.files:
        c, k = key.split("/", 1)
        cases.setdefault(c, {})[k] = npz[key]
    return cases


# ---------------------------------------------------------------------------------------------- voxelizer
def oracle_voxelize_batch(frames, pc_range, voxel_size, max_points, max_voxels):
    """Per-frame oracle voxelization + collate (dataset.py L171-178): voxels, coords [b,z,y,x], num, counts."""
    vs, cs, ns, counts = [], [], [], []
    for b, pts in enumerate(frames):
        g = OV.Point2VoxelCPU3d(voxel_size, pc_range, pts.shape[1], max_points, max_voxels)
        v, c, n = [t.numpy() for t in g.point_to_voxel(OV.from_numpy(pts))]
        vs.append(v)
        ns.append(n)
        cs.append(np.pad(c, ((0, 0), (1, 0)), mode="constant", constant_values=b))
        counts.append(v.shape[0])
    return np.concatenate(vs), np.concatenate(cs).astype(np.int32), np.concatenate(ns), np.array(counts + [sum(counts)])


def canonical_order(coords):
    c = np.asarray(coords)
    return np.lexsort((c[:, 3], c[:, 2], c[:, 1], c[:, 0]))


def gpu_voxelize_batch(frames, pc_range, voxel_size, max_points, max_voxels, order, device="cuda"):
    from toda_b200 import ops
    offs = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)
    f = frames[0].shape[1]
    allp = np.concatenate(frames) if sum(x.shape[0] for x in frames) else np.zeros((0, f), np.float32)
    pts = torch.from_numpy(np.ascontiguousarray(allp)).to(device)
    v, c, n, counts = ops.voxelize(pts, torch.from_numpy(offs).to(device), pc_range, voxel_size, max_points, max_voxels,
                                   num_features=f, order=order)
    return v.cpu().numpy(), c.cpu().numpy(), n.cpu().numpy(), counts.cpu().numpy()


def assert_voxels_equal(got, want, exact_order):
    gv, gc, gn, gcnt = got
    wv, wc, wn, wcnt = want
    assert np.array_equal(gcnt, wcnt), (gcnt, wcnt)
    if not exact_order:
        go, wo = canonical_order(gc), canonical_order(wc)
        gv, gc, gn, wv, wc, wn = gv[go], gc[go], gn[go], wv[wo], wc[wo], wn[wo]
    assert np.array_equal(gc, wc), "voxel coords differ"
    assert np.array_equal(gn, wn), "per-voxel point counts differ"
    assert np.array_equal(gv.view(np.uint32), wv.view(np.uint32)), "point membership / order inside voxels differs"


# ---------------------------------------------------------------------------------------------- rulebooks
def table_to_canonical_pairs(nbr, in_coords, out_coords, in_shape, out_shape):
    """Neighbour table (kvol, n_out) -> sorted (k, out_key, in_key) rows, comparable with
    oracle.spconv_oracle.rulebook_pairs_canonical."""
    nbr = np.asarray(nbr)
    pairs = []
    for k in range(nbr.shape[0]):
        out_rows = np.nonzero(nbr[k] >= 0)[0]
        pairs.append((nbr[k][out_rows].astype(np.int64), out_rows.astype(np.int64)))
    return S.rulebook_pairs_canonical(in_coords, out_coords, pairs, in_shape, out_shape)


def random_sparse(seed, batch, shape, n, c):
    rng = np.random.default_rng(seed)
    d, h, w = shape
    cells = np.sort(rng.choice(batch * d * h * w, size=n, replace=False))
    b = cells // (d * h * w)
    r = cells % (d * h * w)
    idx = np.stack([b, r // (h * w), (r % (h * w)) // w, r % w], axis=1).astype(np.int32)
    feats = rng.standard_normal((n, c)).astype(np.float32)
    return feats, idx


def assert_close(a, b, rtol=RTOL, atol_scale=1e-5, what=""):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    scale = max(np.abs(b).max(), 1e-30) if b.size else 1.0
    err = np.abs(a - b)
    tol = rtol * np.abs(b) + atol_scale * scale
    bad = err > tol
    assert not bad.any(), f"{what}: {bad.sum()} / {bad.size} outside rtol={rtol}; max err {err.max():.3e} (scale {scale:.3e})"


# ---------------------------------------------------------------------------------------------- backbones
def build_pair(name, input_channels, grid_size, seed=666, device="cuda"):
    """(oracle twin on CPU, CUDA plugin) with identical parameters."""
    import toda_b200.pcdet_plugin as P
    torch.manual_seed(seed)
    twin = oracle_backbones()[name](Cfg(), input_channels, np.asarray(grid_size))
    net = getattr(P, name)(Cfg(), input_channels, np.asarray(grid_size)).to(device)
    net.load_state_dict(twin.state_dict())
    return twin, net


def run_backbone(net, hc, voxel_features, voxel_coords, batch_size, cot=None, train=True):
    """fwd (+ bwd with a fixed cotangent on spatial_features).  Returns dict of numpy results."""
    net.train(train)
    vf = voxel_features.clone().requires_grad_(train)
    bd = hc(net({"voxel_features": vf, "voxel_coords": voxel_coords, "batch_size": batch_size}))
    sf = bd["spatial_features"]
    out = {"spatial_features": sf.detach().cpu().numpy(), "enc_features": bd["encoded_spconv_tensor"].features.detach().cpu().numpy(),
           "enc_indices": bd["encoded_spconv_tensor"].indices.cpu().numpy()}
    for k, t in bd["multi_scale_3d_features"].items():
        out[k + "_features"] = t.features.detach().cpu().numpy()
        out[k + "_indices"] = t.indices.cpu().numpy()
    if train:
        loss = (sf * cot.to(sf.device)).sum()
        loss.backward()
        out["loss"] = float(loss.item())
        out["dvoxel_features"] = vf.grad.cpu().numpy()
        out["grads"] = {n: p.grad.detach().cpu().numpy() for n, p in net.named_parameters()}
    return out


def sort_rows(features, indices):
    o = canonical_order(indices)
    return features[o], indices[o]


def run_smoke():
    """Small end-to-end check used by __graft_entry__.smoke()."""
    import toda_b200.pcdet_plugin as P
    from toda_b200 import ops, synth
    dev = "cuda:0"
    pcr, vs, k, mv = [4.0, -2.4, -5.0, 8.8, 2.4, 3.0], [0.075, 0.075, 0.2], 10, 4000
    frames = [synth.make_frame("nus_0075", i) for i in range(2)]
    frames = [f[(f[:, 0] > 3.5) & (f[:, 0] < 9.3) & (np.abs(f[:, 1]) < 2.9)] for f in frames]
    want = oracle_voxelize_batch(frames, pcr, vs, k, mv)
    got = gpu_voxelize_batch(frames, pcr, vs, k, mv, ops.ORDER_FIRST_APPEARANCE, dev)
    assert_voxels_equal(got, want, exact_order=True)
    got_c = gpu_voxelize_batch(frames, pcr, vs, k, mv, ops.ORDER_CANONICAL, dev)
    assert_voxels_equal(got_c, want, exact_order=False)
    grid = ops.grid_size_xyz(pcr, vs)
    twin, net = build_pair("VoxelResBackBone8x", 5, grid, device=dev)
    hc_o = lambda bd: _oracle_hc(bd)  # noqa: E731
    hc_g = P.HeightCompression(Cfg(NUM_BEV_FEATURES=256))
    v, c, n, _ = want
    vf = torch.from_numpy(OV.mean_vfe(v, n))
    vc = torch.from_numpy(c).float()
    gen = torch.Generator().manual_seed(1)
    ro = run_backbone(twin, hc_o, vf, vc, 2, cot=None, train=False)
    cot = torch.randn(ro["spatial_features"].shape, generator=gen)
    ro = run_backbone(twin, hc_o, vf, vc, 2, cot=cot, train=True)
    gv = ops.mean_vfe(torch.from_numpy(v).to(dev), torch.from_numpy(n).to(dev))
    assert_close(gv.cpu().numpy(), vf.numpy(), what="MeanVFE")
    rg = run_backbone(net, hc_g, gv.detach(), vc.to(dev), 2, cot=cot, train=True)
    assert np.array_equal(*[sort_rows(r["enc_features"], r["enc_indices"])[1] for r in (rg, ro)])
    assert_close(rg["spatial_features"], ro["spatial_features"], what="spatial_features")
    assert_close(rg["dvoxel_features"], ro["dvoxel_features"], rtol=1e-3, what="d voxel_features")
    gmax = max(float(np.abs(g).max()) for g in ro["grads"].values())
    for name, g in ro["grads"].items():
        # conv biases in front of a BatchNorm have a mathematically zero gradient (rounding noise ~1e-7 of the
        # weight gradients): compare those on the global gradient scale
        if name.endswith(".bias") and float(np.abs(g).max()) < 1e-5 * gmax:
            assert float(np.abs(rg["grads"][name]).max()) < 1e-5 * gmax, name
        else:
            assert_close(rg["grads"][name], g, rtol=1e-3, atol_scale=1e-4, what="grad " + name)
    # the same step on the bf16 tensor-core path (what bench.py times): the tcgen05 forward / dgrad / wgrad kernels run,
    # geometry stays bit-identical, activations within the stated bf16 tolerance (relative L2 <= 5e-2) of the oracle
    from toda_b200.spconv_compat import pytorch as G
    _, net_b = build_pair("VoxelResBackBone8x", 5, grid, device=dev)
    for plans in (False, True):                 # round-1 kernels, then the row-cache / TMEM-operand kernel
        ops.set_tile_plans(plans)
        G.set_conv_precision("bf16")
        try:
            rb = run_backbone(net_b, hc_g, gv.detach(), vc.to(dev), 2, cot=cot, train=True)
        finally:
            G.set_conv_precision("fp32")
            ops.set_tile_plans(False)
        assert np.array_equal(sort_rows(rb["enc_features"], rb["enc_indices"])[1], sort_rows(ro["enc_features"], ro["enc_indices"])[1])
        a, b = rb["spatial_features"].astype(np.float64), ro["spatial_features"].astype(np.float64)
        rel = float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
        assert rel <= 5e-2, ("bf16 spatial_features rel-L2", rel)


def _oracle_hc(bd):
    t = bd["encoded_spconv_tensor"]
    d = t.dense()
    n, c, dd, h, w = d.shape
    bd["spatial_features"] = d.view(n, c * dd, h, w)
    bd["spatial_features_stride"] = bd["encoded_spconv_tensor_stride"]
    return bd
