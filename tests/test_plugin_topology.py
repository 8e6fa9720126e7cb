"""Host-logic tests (CPU): the plugin's declarative backbone topology, instantiated on the CPU oracle
provider, reproduces the golden vectors that were generated through the REFERENCE'S OWN
spconv_backbone.py / height_compression.py (tests/golden/make_golden.py) -- same parameter names, same
init order, same outputs and gradients."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU


@pytest.mark.parametrize("cls,fname", [("VoxelResBackBone8x", "backbone_res.npz"), ("VoxelBackBone8x", "backbone_voxel.npz"),
                                       ("VoxelResBackBone8x", "backbone_res_stage2.npz")])
def test_twin_reproduces_reference_golden(cls, fname):
    g = PU.load_golden(fname)
    torch.manual_seed(int(g["seed"]))
    net = PU.oracle_backbones()[cls](PU.Cfg(), int(g["voxel_features"].shape[1]), g["grid_size"])
    if "stage2" in fname:      # TODA stage-1/2 grid: 49 z bins -> sparse_shape 50 -> 25 -> 13 -> 6 -> 2
        assert list(net.sparse_shape)[0] == 50
    wsum = float(sum(p.detach().double().abs().sum() for p in net.parameters()))
    assert abs(wsum - float(g["weight_abs_sum"])) < 1e-6 * wsum      # identical init => identical param order
    vf, vc = torch.from_numpy(g["voxel_features"]), torch.from_numpy(g["voxel_coords"]).float()
    gen = torch.Generator().manual_seed(int(g["seed"]))
    cot = torch.randn(tuple(g["bev_shape"]), generator=gen)
    with PU.golden_threads():
        r = PU.run_backbone(net, PU._oracle_hc, vf, vc, 2, cot=cot, train=True)
    assert np.array_equal(r["enc_indices"], g["train_enc_indices"])
    np.testing.assert_allclose(r["enc_features"], g["train_enc_features"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(r["dvoxel_features"], g["train_dvoxel_features"], rtol=1e-4, atol=1e-6)
    assert abs(r["loss"] - float(g["train_loss"])) < 1e-3
    names = [str(n) for n in g["grad_names"]]
    assert names == [n for n, _ in net.named_parameters()]
    norms = np.array([np.linalg.norm(r["grads"][n].astype(np.float64)) for n in names])
    np.testing.assert_allclose(norms, g["grad_norms"], rtol=1e-3, atol=1e-5)
    for k in ["x_conv1", "x_conv2", "x_conv3", "x_conv4"]:
        assert np.array_equal(r[k + "_indices"], g[f"train_{k}_indices"])
        np.testing.assert_allclose(r[k + "_features"], g[f"train_{k}_features"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("cls,fname", [("VoxelResBackBone8x", "backbone_res.npz"), ("VoxelBackBone8x", "backbone_voxel.npz")])
def test_cuda_plugin_parameters_match_reference_golden(cls, fname):
    """The CUDA plugin module (constructed on the CPU) has the reference's parameter names, order and seeded initial
    values, as recorded in the golden built through the reference's own spconv_backbone.py."""
    import toda_b200.pcdet_plugin as P
    g = PU.load_golden(fname)
    torch.manual_seed(int(g["seed"]))
    net = getattr(P, cls)(PU.Cfg(), int(g["voxel_features"].shape[1]), g["grid_size"])
    assert [n for n, _ in net.named_parameters()] == [str(n) for n in g["grad_names"]]
    wsum = float(sum(p.detach().double().abs().sum() for p in net.parameters()))
    assert abs(wsum - float(g["weight_abs_sum"])) < 1e-6 * wsum
    assert net.conv_input[0].weight.shape == g["grad_conv_input_weight"].shape
    assert net.conv_out[0].weight.shape == g["grad_conv_out_weight"].shape


def test_state_dict_matches_reference_when_present():
    from oracle import reference_loader as R, spconv_oracle as S
    if not R.available():
        pytest.skip("needs a rasd3/TODA checkout named by TODA_REFERENCE")
    ns = R.load(S.make_modules())
    for cls in ["VoxelResBackBone8x", "VoxelBackBone8x"]:
        ref = getattr(ns, cls)(R.Cfg(), 5, np.array([1440, 1440, 40]))
        mine = PU.oracle_backbones()[cls](PU.Cfg(), 5, np.array([1440, 1440, 40]))
        a = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
        b = {k: tuple(v.shape) for k, v in mine.state_dict().items()}
        assert a == b
        assert list(ref.sparse_shape) == list(mine.sparse_shape) == [41, 1440, 1440]
        assert ref.num_point_features == mine.num_point_features and ref.backbone_channels == mine.backbone_channels


def test_golden_voxelizer_fixture_matches_oracle():
    """The committed voxelizer goldens (produced through the reference's data_processor.py) equal what the C
    oracle gives on the recorded points -- guards fixture / oracle drift."""
    from oracle import voxelize as OV
    cases = PU.golden_cases(PU.load_golden("voxelize.npz"))
    assert set(cases) == {"crop_nus", "crop_nus_capped", "crop_waymo", "coarse_full_nus"}
    for name, c in cases.items():
        g = OV.Point2VoxelCPU3d(c["voxel_size"], c["pc_range"], c["points"].shape[1], int(c["max_points"]), int(c["max_voxels"]))
        v, co, n = [t.numpy() for t in g.point_to_voxel(OV.from_numpy(c["points"]))]
        assert np.array_equal(v, c["voxels"]) and np.array_equal(co, c["voxel_coords"]) and np.array_equal(n, c["voxel_num_points"])
        assert list(g.grid) == list(c["grid_size"])
        np.testing.assert_allclose(OV.mean_vfe(v, n), c["voxel_features"], rtol=1e-6, atol=1e-7)
    assert cases["crop_nus_capped"]["voxels"].shape[0] == 700      # the max_voxels cap is active in this case


def test_point_preprocessor_two_phase_protocol_on_cpu():
    """Construction binds the configured steps in order and publishes grid_size / voxel_size like the reference's
    DataProcessor (data_processor.py L64-76, L105-113); no CUDA call is made until a batch is processed."""
    import pytest
    from toda_b200.pcdet_plugin.processor import PointPreprocessor
    from tests.parity_utils import Cfg
    cfgs = [Cfg(NAME="mask_points_and_boxes_outside_range", REMOVE_OUTSIDE_BOXES=True),
            Cfg(NAME="shuffle_points", SHUFFLE_ENABLED=Cfg(train=True, test=False)),
            Cfg(NAME="transform_points_to_voxels_placeholder", VOXEL_SIZE=[0.075, 0.075, 0.2])]
    pp = PointPreprocessor(cfgs, np.array([-54.0, -54.0, -5.0, 54.0, 54.0, 3.0], np.float32), training=False, num_point_features=5)
    assert pp.grid_size.tolist() == [1440, 1440, 40] and pp.voxel_size == [0.075, 0.075, 0.2] and pp.mode == "test"
    assert len(pp.data_processor_queue) == 3
    # shuffle disabled in test mode: the bound step returns the dict untouched (no device work)
    marker = object()
    assert pp.data_processor_queue[1](data_dict={"points": marker})["points"] is marker
    with pytest.raises(NotImplementedError):
        PointPreprocessor([Cfg(NAME="transform_points_to_voxels", VOXEL_SIZE=[0.1, 0.1, 0.2])], np.zeros(6, np.float32), True, 5)


def test_box_params_packing_is_host_logic():
    """K0 box mode parameters: count, margin, then seven float32 values per box; extra gt_boxes columns are dropped."""
    import numpy as np
    import torch
    from toda_b200.pcdet_plugin.processor import _box_params
    b = np.arange(16, dtype=np.float32).reshape(2, 8)
    want = [2.0, float(np.float32(0.1))] + [0, 1, 2, 3, 4, 5, 6, 8, 9, 10, 11, 12, 13, 14]
    got = _box_params(b, np.float32(0.1))
    assert got == [float(v) for v in want]
    assert _box_params(torch.from_numpy(b), np.float32(0.1)) == got
    assert _box_params(b[:0], 0.1) == [0.0, 0.1]
