"""The REFERENCE'S OWN files bound against toda_b200's drop-in `spconv` / `cumm` modules (CPU: construction and
parameter plumbing only, no kernels): `spconv_backbone.py` builds both backbones on `toda_b200.spconv_compat`,
state_dict keys / shapes equal the plugin's, `find_all_spconv_keys` (pcdet/utils/spconv_utils.py L11-26) finds every
conv weight, and the checkpoint re-layout of `Detector3DTemplate._load_state_dict`
(pcdet/models/detectors/detector3d_template.py L330-357) loads spconv-1.x / transposed weights into the plugin modules.
The tests that load the reference's files need a rasd3/TODA checkout named by TODA_REFERENCE and skip without one; the
checkpoint re-layout runs without it and is cross-checked against the reference's loader when it is there."""
import numpy as np
import pytest
import torch

from tests import parity_utils as PU


def _ref():
    from oracle import reference_loader as R
    if not R.available():
        pytest.skip("needs a rasd3/TODA checkout named by TODA_REFERENCE")
    import toda_b200.spconv_compat as sc
    return R, R.load(sc.make_modules())


def _spconv_weight_keys(net):
    """What find_all_spconv_keys (pcdet/utils/spconv_utils.py L11-26) returns: the weight key of every sparse conv."""
    from toda_b200.spconv_compat import pytorch as G
    return {name + ".weight" for name, m in net.named_modules() if isinstance(m, G.SparseConvolution)}


@pytest.mark.parametrize("cls,nconv", [("VoxelResBackBone8x", 21), ("VoxelBackBone8x", 12)])
def test_reference_backbone_builds_on_the_cuda_shim(cls, nconv):
    R, ns = _ref()
    import toda_b200.pcdet_plugin as P
    from toda_b200.spconv_compat import pytorch as G
    torch.manual_seed(666)
    ref = getattr(ns, cls)(R.Cfg(), 5, np.array([1440, 1440, 40]))
    torch.manual_seed(666)
    mine = getattr(P, cls)(PU.Cfg(), 5, np.array([1440, 1440, 40]))
    convs = [m for m in ref.modules() if isinstance(m, G.SparseConvolution)]
    assert len(convs) == nconv
    a = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    b = {k: tuple(v.shape) for k, v in mine.state_dict().items()}
    assert a == b                                                # same parameter names and shapes
    for k, v in ref.state_dict().items():                        # same init order => same values under one seed
        assert torch.equal(v, mine.state_dict()[k]), k
    keys = ns.spconv_utils.find_all_spconv_keys(ref)
    assert len(keys) == nconv and all(k.endswith(".weight") for k in keys)
    assert keys == ns.spconv_utils.find_all_spconv_keys(mine)
    assert list(ref.sparse_shape) == list(mine.sparse_shape) == [41, 1440, 1440]
    # the reference's replace_feature helper takes the spconv-2.x branch on our tensor type
    t = G.SparseConvTensor(torch.zeros(3, 4), torch.zeros(3, 4, dtype=torch.int32), [4, 4, 4], 1)
    t2 = ns.spconv_utils.replace_feature(t, torch.ones(3, 4))
    assert t2 is not t and float(t2.features.sum()) == 12.0 and t2.indices is t.indices


def _load_state_dict_like_reference(model, model_state_disk, spconv_keys):
    """Restatement for the test of detector3d_template.py L330-357 (the method lives on Detector3DTemplate, which cannot be
    constructed without the rest of pcdet): same shape tests, same two layout conversions."""
    state_dict = model.state_dict()
    update = {}
    for key, val in model_state_disk.items():
        if key in spconv_keys and key in state_dict and state_dict[key].shape != val.shape:
            val_native = val.transpose(-1, -2)
            if val_native.shape == state_dict[key].shape:
                val = val_native.contiguous()
            else:
                assert len(val.shape) == 5
                val_implicit = val.permute(4, 0, 1, 2, 3)
                if val_implicit.shape == state_dict[key].shape:
                    val = val_implicit.contiguous()
        if key in state_dict and state_dict[key].shape == val.shape:
            update[key] = val
    state_dict.update(update)
    model.load_state_dict(state_dict)
    return update


def test_checkpoint_relayout_from_spconv1_weights():
    """A checkpoint written with spconv 1.x holds conv weights as (kz,ky,kx,Cin,Cout); the reference loader permutes them
    to the layout of the running spconv.  The plugin's layout (Cout,kz,ky,kx,Cin) must be reached by its `val_implicit`
    branch for every conv, and the permuted weights must be the same convolution."""
    import inspect
    import os
    import toda_b200.pcdet_plugin as P
    from oracle import reference_loader as R
    torch.manual_seed(1)
    net = P.VoxelResBackBone8x(PU.Cfg(), 5, np.array([1440, 1440, 40]))
    keys = _spconv_weight_keys(net)
    assert len(keys) == 21
    if R.available():         # the two restatements of this test are the reference's own code
        import toda_b200.spconv_compat as sc
        ns = R.load(sc.make_modules())
        src = open(os.path.join(R.REF_ROOT, "pcdet/models/detectors/detector3d_template.py")).read()
        assert "val.permute(4, 0, 1, 2, 3)" in src and "val.transpose(-1, -2)" in src
        assert ns.spconv_utils.find_all_spconv_keys(net) == keys
    want = {k: v.clone() for k, v in net.state_dict().items()}
    disk = {}
    for k, v in want.items():
        disk[k] = v.permute(1, 2, 3, 4, 0).contiguous() if k in keys else v.clone()      # (Cout,kz,ky,kx,Cin) -> (kz,ky,kx,Cin,Cout)
    torch.manual_seed(2)
    fresh = P.VoxelResBackBone8x(PU.Cfg(), 5, np.array([1440, 1440, 40]))
    update = _load_state_dict_like_reference(fresh, disk, keys)
    assert set(update) == set(want)                               # nothing was dropped for a shape mismatch
    for k, v in fresh.state_dict().items():
        assert torch.equal(v, want[k]), k
    # square layers (Cin == Cout, e.g. 16->16): the first shape test of the loader (transpose(-1,-2)) must NOT fire for a
    # 1.x tensor, or the weights would be silently scrambled: (3,3,3,16,16) != (16,3,3,3,16) keeps it out
    k16 = [k for k in keys if want[k].shape == (16, 3, 3, 3, 16)][0]
    assert disk[k16].transpose(-1, -2).shape != want[k16].shape
    assert inspect.isclass(P.VoxelResBackBone8x)
