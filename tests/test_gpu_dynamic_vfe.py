"""DynamicMeanVFE on the GPU (ops.voxelize_dynamic, pcdet_plugin.DynamicMeanVFE) against the restatement in
tests/dynamic_vfe_oracle.py: features, coords and per-frame counts bit for bit after canonical sorting."""
import ctypes
import types

import numpy as np
import pytest
import torch

from tests import dynamic_vfe_oracle as DV
from tests import parity_utils as PU

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _collate(frames):
    cols = [np.pad(f, ((0, 0), (1, 0)), constant_values=b) for b, f in enumerate(frames)]
    stride = 1 + (frames[0].shape[1] if frames else 4)
    pts = np.concatenate(cols) if sum(f.shape[0] for f in frames) else np.zeros((0, stride), np.float32)
    offs = np.cumsum([0] + [f.shape[0] for f in frames]).astype(np.int32)
    return np.ascontiguousarray(pts, np.float32), offs


def _check(frames, pcr, vs, grid=None):
    from toda_b200 import ops
    grid = ops.grid_size_xyz(pcr, vs) if grid is None else np.asarray(grid)
    pts, offs = _collate(frames)
    f, c, n = ops.voxelize_dynamic(torch.from_numpy(pts).to(DEV), torch.from_numpy(offs).to(DEV), pcr, vs, grid=grid)
    wf, wc, wn = DV.dynamic_mean_vfe(pts, len(frames), pcr, vs, grid)
    wf, wc = DV.canonical(wf, wc)
    f, c, n = f.cpu().numpy(), c.cpu().numpy(), n.cpu().numpy()
    assert np.array_equal(n, wn), (n, wn)
    assert np.array_equal(c, wc), "coords differ"
    bad = np.nonzero((f.view(np.uint32) != wf.view(np.uint32)).any(axis=1))[0]
    assert bad.size == 0, f"features differ in {bad.size} of {f.shape[0]} voxels, first {c[bad[:4]].tolist()}: " \
                          f"{f[bad[:2]].tolist()} != {wf[bad[:2]].tolist()}"
    return f, c, n


@pytest.mark.parametrize("config", ["nus_0075", "waymo_010", "toda_stage2"])
def test_full_batches_are_bit_exact(config):
    from toda_b200 import synth
    cfg = synth.CONFIGS[config]
    frames, _ = synth.make_batch(config, 4)
    pcr = list(cfg["pc_range"])
    if config == "toda_stage2":
        assert frames[0].shape[1] == 4 and pcr[5] == 4.8
    _, _, n = _check(frames, pcr, cfg["voxel_size"])
    assert n[4] > 10000


def test_empty_batch_frames_and_out_of_range():
    from toda_b200 import synth
    cfg = synth.CONFIGS["nus_0075"]
    pcr, vs = cfg["pc_range"], cfg["voxel_size"]
    a, b = synth.make_frame("nus_0075", 1), synth.make_frame("nus_0075", 2)
    empty = np.zeros((0, 5), np.float32)
    one = a[:1].copy()
    outside = a[:500].copy()
    outside[:, 0] += 200.0
    _, _, n = _check([empty, empty], pcr, vs)
    assert n.tolist() == [0, 0, 0]
    _, _, n = _check([a, empty, b], pcr, vs)
    assert n[1] == 0 and n[0] > 0 and n[2] > 0
    _, _, n = _check([one, a, outside], pcr, vs)
    assert n[0] == 1 and n[2] == 0


def test_nan_rows_and_boundary_points():
    pcr, vs = [-4.0, -4.0, -2.0, 4.0, 4.0, 2.0], [0.5, 0.5, 0.25]
    rng = np.random.default_rng(5)
    pts = rng.uniform(-4.5, 4.5, (20000, 4)).astype(np.float32)
    pts[:, 2] = rng.uniform(-2.5, 2.5, 20000)
    pts[::97, 0] = np.nan
    pts[1::89, 2] = np.nan
    lo, hi = np.float32(pcr[:3]), np.float32(pcr[3:])
    pts[2::50, :3] = lo                     # on lo: kept
    pts[3::50, 0] = hi[0]                   # quotient exactly grid on x: dropped
    pts[4::50, 2] = hi[2]                   # on z: dropped
    pts[5::50, 2] = np.nextafter(hi[2], np.float32(0))
    _check([pts[:12000], pts[12000:]], pcr, vs)


def test_one_voxel_with_100000_points():
    from toda_b200 import synth
    cfg = synth.CONFIGS["nus_0075"]
    rng = np.random.default_rng(9)
    heavy = np.zeros((100000, 5), np.float32)
    heavy[:, :3] = rng.uniform(1.06, 1.12, (100000, 3))     # one cell of the 0.075 m grid: x, y index 734
    heavy[:, 2] = rng.uniform(0.0, 0.19, 100000)
    heavy[:, 3:] = rng.standard_normal((100000, 2))
    f, c, n = _check([synth.make_frame("nus_0075", 3), heavy, synth.make_frame("nus_0075", 4)], cfg["pc_range"],
                     cfg["voxel_size"])
    assert n[1] == 1


@pytest.mark.parametrize("stride", [4, 5, 12, 47])
def test_strides(stride):
    rng = np.random.default_rng(stride)
    pcr, vs = [-10.0, -10.0, -3.0, 10.0, 10.0, 3.0], [0.2, 0.2, 0.5]
    fr = []
    for b in range(3):
        p = rng.standard_normal((30000, stride - 1)).astype(np.float32)
        p[:, :3] *= np.float32([4.0, 4.0, 1.0])
        fr.append(p)
    _check(fr, pcr, vs)


def test_run_to_run_bit_equality_and_agreement_with_hard_voxelizer():
    from toda_b200 import ops, synth
    cfg = synth.CONFIGS["nus_0075"]
    frames, collated = synth.make_batch("nus_0075", 2)
    pts = torch.from_numpy(collated).to(DEV)
    offs = torch.tensor(np.cumsum([0] + [f.shape[0] for f in frames]), dtype=torch.int32, device=DEV)
    runs = [ops.voxelize_dynamic(pts, offs, cfg["pc_range"], cfg["voxel_size"]) for _ in range(3)]
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)
    f, c, n = runs[0]
    pts1, offs1 = pts[: frames[0].shape[0]].contiguous(), offs[:2].contiguous()
    f1, c1, _ = ops.voxelize_dynamic(pts1, offs1, cfg["pc_range"], cfg["voxel_size"])
    # K = the largest voxel of the frame, max_voxels = N: no cap binds, so hard voxelization + MeanVFE is the same mean
    kmax = int(_max_count(pts1.cpu().numpy(), cfg))
    assert kmax > 1
    v, hc, num, _ = ops.voxelize(pts1, offs1, cfg["pc_range"], cfg["voxel_size"], kmax, pts1.shape[0], xyz_col=1, feat_col=1,
                                 order=ops.ORDER_CANONICAL)
    assert torch.equal(hc, c1) and torch.equal(ops.mean_vfe(v, num), f1)


def _max_count(pts, cfg):
    from toda_b200 import ops
    lo, vs = np.float32(cfg["pc_range"][:3]), np.float32(cfg["voxel_size"])
    grid = ops.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    with np.errstate(invalid="ignore"):
        q = np.floor((pts[:, 1:4] - lo) / vs)
    keep = np.all((q >= 0) & (q < grid), axis=1)
    return np.unique(q[keep], axis=0, return_counts=True)[1].max()


def test_index_is_left_clean_for_hard_voxelization_and_rulebooks():
    from toda_b200 import ops, synth
    cfg = synth.CONFIGS["nus_0075"]
    frames, collated = synth.make_batch("nus_0075", 2, first_frame=5)
    pts = torch.from_numpy(collated).to(DEV)
    offs = torch.tensor(np.cumsum([0] + [f.shape[0] for f in frames]), dtype=torch.int32, device=DEV)
    pcr, vs = cfg["pc_range"], cfg["voxel_size"]

    def hard_and_rulebook(tag):
        v, c, num, cnt = ops.voxelize(pts, offs, pcr, vs, 10, 120000, xyz_col=1, feat_col=1, order=ops.ORDER_CANONICAL)
        grid = ops.grid_size_xyz(pcr, vs)
        index = ops.OccupancyIndex(2, [int(grid[2]), int(grid[1]), int(grid[0])], DEV, tag)
        index.insert(c)
        built = index.build(c.shape[0])
        rb = ops.rulebook_subm(index, [3, 3, 3])
        out = [t.clone() for t in (v, c, num, cnt, built, rb.nbr_fwd)]
        index.release()
        return out

    fresh = hard_and_rulebook("dyn_a")
    ops.voxelize_dynamic(pts, offs, pcr, vs)
    after = hard_and_rulebook("dyn_b")
    for a, b in zip(fresh, after):
        assert torch.equal(a, b)


def test_argument_errors():
    from toda_b200 import _C, ops
    pts = torch.zeros((10, 5), device=DEV)
    offs = torch.tensor([0, 10], dtype=torch.int32, device=DEV)
    pcr, vs = [0, 0, 0, 1, 1, 1], [0.1, 0.1, 0.1]
    with pytest.raises(TypeError):
        ops.voxelize_dynamic(pts.double(), offs, pcr, vs)
    with pytest.raises(TypeError):
        ops.voxelize_dynamic(pts, offs.long(), pcr, vs)
    with pytest.raises(TypeError):
        ops.voxelize_dynamic(pts.cpu().numpy(), offs, pcr, vs)
    with pytest.raises(ValueError):
        ops.voxelize_dynamic(pts[:, :3].contiguous(), offs, pcr, vs)
    with pytest.raises(ValueError):
        ops.voxelize_dynamic(pts, offs[:1], pcr, vs)
    with pytest.raises(ValueError):
        ops.voxelize_dynamic(pts, offs, pcr, [0.1, 0.0, 0.1])
    with pytest.raises(ValueError):
        ops.voxelize_dynamic(pts, offs, pcr, vs, grid=[10, 10])
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.voxelize_dynamic(pts.cpu(), offs, pcr, vs)
    with pytest.raises(RuntimeError, match="point_stride 48 too large"):
        ops.voxelize_dynamic(torch.zeros((10, 48), device=DEV), offs, pcr, vs)
    # the C entry point itself
    L = _C.lib()
    grid = _C.ints([10, 10, 10])
    rng, vsz = _C.floats(pcr), _C.floats(vs)
    out = torch.empty((10, 4), device=DEV)
    co = torch.empty((10, 4), dtype=torch.int32, device=DEV)
    cnt = torch.empty((2,), dtype=torch.int32, device=DEV)
    nbytes = L.toda_voxelize_dynamic_workspace_bytes(10, 1, grid)
    ws = torch.empty((nbytes,), dtype=torch.uint8, device=DEV)
    p = ctypes.c_void_p
    args = [p(pts.data_ptr()), 10, 5, 1, 1, 4, p(offs.data_ptr()), 1, rng, vsz, grid, p(out.data_ptr()), p(co.data_ptr()),
            p(cnt.data_ptr()), p(ws.data_ptr()), nbytes, None]
    assert L.toda_voxelize_dynamic(*args) == 0
    bad = list(args)
    bad[5] = 5                                      # feat_col + F > stride
    assert L.toda_voxelize_dynamic(*bad) == -1 and b"column layout" in L.toda_last_error()
    bad = list(args)
    bad[15] = nbytes - 1
    assert L.toda_voxelize_dynamic(*bad) != 0 and b"workspace" in L.toda_last_error()
    bad = list(args)
    bad[11] = None
    assert L.toda_voxelize_dynamic(*bad) == -1 and b"null output" in L.toda_last_error()
    assert L.toda_voxelize_dynamic_workspace_bytes(10, 0, grid) == 0


def _stub_pcdet_models():
    reg = lambda: types.SimpleNamespace(__all__={})  # noqa: E731
    return types.SimpleNamespace(backbones_3d=types.SimpleNamespace(vfe=reg(), __all__={}),
                                 backbones_2d=types.SimpleNamespace(map_to_bev=reg()))


def test_register_installs_dynamic_mean_vfe_and_outputs_carry_no_grad():
    import toda_b200.pcdet_plugin as P
    from toda_b200 import synth
    models = _stub_pcdet_models()
    P.register(models)
    cls = models.backbones_3d.vfe.__all__["DynamicMeanVFE"]
    assert cls is P.DynamicMeanVFE
    cfg = synth.CONFIGS["nus_0075"]
    grid = synth.grid_size_xyz(cfg["pc_range"], cfg["voxel_size"])
    vfe = cls(model_cfg=PU.Cfg(NAME="DynamicMeanVFE"), num_point_features=5, voxel_size=cfg["voxel_size"], grid_size=grid,
              point_cloud_range=np.asarray(cfg["pc_range"]), depth_downsample_factor=None)
    assert vfe.get_output_feature_dim() == 5
    frames, collated = synth.make_batch("nus_0075", 2)
    pts = torch.from_numpy(collated).to(DEV).requires_grad_(True)
    bd = vfe({"points": pts, "batch_size": 2})       # no point_frame_offsets: found from the batch column
    assert not bd["voxel_features"].requires_grad and bd["voxel_coords_canonical"] is True
    wf, wc, _ = DV.dynamic_mean_vfe(collated, 2, cfg["pc_range"], cfg["voxel_size"], grid)
    wf, wc = DV.canonical(wf, wc)
    assert np.array_equal(bd["voxel_coords"].cpu().numpy(), wc)
    assert np.array_equal(bd["voxel_features"].cpu().numpy().view(np.uint32), wf.view(np.uint32))


def _crop(frames, pcr):
    return [f[(f[:, 0] > pcr[0] - 0.5) & (f[:, 0] < pcr[3] + 0.5) & (np.abs(f[:, 1]) < pcr[4] + 0.5)] for f in frames]


def test_backbone_chain_matches_oracle_backbone():
    import toda_b200.pcdet_plugin as P
    from toda_b200 import synth
    pcr, vs = [4.0, -2.4, -5.0, 8.8, 2.4, 3.0], [0.075, 0.075, 0.2]
    grid = synth.grid_size_xyz(pcr, vs)
    frames = _crop([synth.make_frame("toda_stage2", i) for i in range(2)], pcr)
    pts, offs = _collate(frames)
    vfe = P.DynamicMeanVFE(PU.Cfg(), 4, vs, grid, pcr)
    bd = vfe({"points": torch.from_numpy(pts).to(DEV), "point_frame_offsets": torch.from_numpy(offs).to(DEV), "batch_size": 2})
    wf, wc, _ = DV.dynamic_mean_vfe(pts, 2, pcr, vs, grid)
    wf, wc = DV.canonical(wf, wc)
    assert np.array_equal(bd["voxel_coords"].cpu().numpy(), wc)
    twin, net = PU.build_pair("VoxelBackBone8x", 4, grid, device=DEV)
    hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
    vf, vc = torch.from_numpy(wf), torch.from_numpy(wc).float()
    ro = PU.run_backbone(twin, PU._oracle_hc, vf, vc, 2, train=False)
    cot = torch.randn(ro["spatial_features"].shape, generator=torch.Generator().manual_seed(1))
    ro = PU.run_backbone(twin, PU._oracle_hc, vf, vc, 2, cot=cot, train=True)
    rg = PU.run_backbone(net, hc, bd["voxel_features"], bd["voxel_coords"], 2, cot=cot, train=True)
    PU.assert_close(rg["spatial_features"], ro["spatial_features"], what="spatial_features")
    PU.assert_close(rg["dvoxel_features"], ro["dvoxel_features"], rtol=1e-3, what="d voxel_features")
    gmax = max(float(np.abs(g).max()) for g in ro["grads"].values())
    for name, g in ro["grads"].items():
        if name.endswith(".bias") and float(np.abs(g).max()) < 1e-5 * gmax:
            assert float(np.abs(rg["grads"][name]).max()) < 1e-5 * gmax, name
        else:
            PU.assert_close(rg["grads"][name], g, rtol=1e-3, atol_scale=1e-4, what="grad " + name)


def test_input_pipeline_equals_inline():
    import toda_b200.pcdet_plugin as P
    from toda_b200 import synth
    from toda_b200.pipeline import InputPipeline
    pcr = [0.0, -9.6, -5.0, 19.2, 9.6, 3.0]
    vs = synth.CONFIGS["nus_0075"]["voxel_size"]
    grid = synth.grid_size_xyz(pcr, vs)
    torch.manual_seed(666)
    vfe = P.DynamicMeanVFE(PU.Cfg(), 5, vs, grid, pcr)
    net = P.VoxelResBackBone8x(PU.Cfg(), 5, grid).to(DEV).train()
    hc = P.HeightCompression(PU.Cfg(NUM_BEV_FEATURES=256))
    host = [_collate(_crop([synth.make_frame("nus_0075", 10 * j + b) for b in range(2)], pcr)) for j in range(2)]

    def run(bd):
        net.zero_grad(set_to_none=True)
        out = hc(net(bd))
        sf = out["spatial_features"]
        cot = torch.randn(sf.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
        (sf * cot).sum().backward()
        return sf.detach().clone(), {n: p.grad.detach().clone() for n, p in net.named_parameters()}

    state = {k: v.clone() for k, v in net.state_dict().items()}
    want = [run(vfe({"points": torch.from_numpy(p).to(DEV), "point_frame_offsets": torch.from_numpy(o).to(DEV),
                     "batch_size": 2})) for p, o in host]
    net.load_state_dict(state)
    pipe = InputPipeline(vfe, net, DEV, reserve_bytes=64 << 20)
    h = pipe.submit({"points": torch.from_numpy(host[0][0]).pin_memory(),
                     "point_frame_offsets": torch.from_numpy(host[0][1]).pin_memory(), "batch_size": 2})
    for i in range(2):
        bd = pipe.consume(h)
        assert "spconv_geometry" in bd
        if i + 1 < 2:
            h = pipe.submit({"points": torch.from_numpy(host[1][0]).pin_memory(),
                             "point_frame_offsets": torch.from_numpy(host[1][1]).pin_memory(), "batch_size": 2})
        sf, grads = run(bd)
        assert torch.equal(sf, want[i][0])
        for name in grads:
            assert torch.equal(grads[name], want[i][1][name]), name
    torch.cuda.synchronize()
