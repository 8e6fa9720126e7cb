"""oracle/reference_loader.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Loads the reference's OWN hot-path Python files by file path (SURVEY.md Appendix B) so that
golden vectors can be produced through them.  `import pcdet` cannot work as shipped
(pcdet/datasets/__init__.py L39-40 is a SyntaxError; easydict / SharedArray / skimage /
compiled ops are absent), so a synthetic package skeleton is created and only these files run:
    pcdet/utils/common_utils.py, pcdet/utils/box_utils.py,
    pcdet/ops/roiaware_pool3d/roiaware_pool3d_utils.py,
    pcdet/datasets/processor/data_processor.py,
    pcdet/utils/spconv_utils.py,
    pcdet/models/backbones_3d/vfe/{vfe_template,mean_vfe}.py,
    pcdet/models/backbones_2d/map_to_bev/height_compression.py,
    pcdet/models/backbones_3d/spconv_backbone.py
The arithmetic they call (`spconv`, `cumm`) is supplied by a provider: the CPU oracle
(oracle.spconv_oracle.make_modules()) when generating goldens.

The reference is a checkout of rasd3/TODA named by the TODA_REFERENCE environment variable; it is not part of
this repository.  Nothing that runs under `-m gpu`, smoke() or bench.py may call this, and the tests that need it
skip when TODA_REFERENCE is unset.
"""
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("TODA_REFERENCE", "")


class Cfg(dict):
    """EasyDict stand-in: attribute access + .get (Appendix B step 5)."""
    __getattr__ = dict.get

    def __setattr__(self, k, v):
        self[k] = v


def available(root=REF_ROOT):
    return bool(root) and os.path.isfile(os.path.join(root, "pcdet/models/backbones_3d/spconv_backbone.py"))


def _pkg(name, path=None):
    m = types.ModuleType(name)
    m.__path__ = [path] if path else []
    sys.modules[name] = m
    return m


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    parent, _, leaf = name.rpartition(".")
    if parent in sys.modules:
        setattr(sys.modules[parent], leaf, mod)
    return mod


def load(provider_modules, root=REF_ROOT):
    """Returns a namespace with the reference's classes bound against `provider_modules`
    (a dict name->module containing at least spconv, spconv.pytorch, spconv.pytorch.conv,
    spconv.utils, cumm, cumm.tensorview)."""
    if not available(root):
        raise FileNotFoundError(root)
    # drop any earlier load so that the reference files re-bind to this provider
    for k in [k for k in sys.modules if k == "pcdet" or k.startswith("pcdet.")]:
        del sys.modules[k]
    sys.modules.update(provider_modules)
    P = os.path.join(root, "pcdet")
    for name in ["pcdet", "pcdet.utils", "pcdet.ops", "pcdet.ops.roiaware_pool3d", "pcdet.datasets",
                 "pcdet.datasets.processor", "pcdet.models", "pcdet.models.backbones_3d",
                 "pcdet.models.backbones_3d.vfe", "pcdet.models.backbones_2d",
                 "pcdet.models.backbones_2d.map_to_bev"]:
        _pkg(name)
        parent, _, leaf = name.rpartition(".")
        if parent:
            setattr(sys.modules[parent], leaf, sys.modules[name])
    # stubs for absent third-party / compiled modules that the files import but the hot path never calls
    for stub in ["SharedArray", "skimage", "skimage.transform"]:
        if stub not in sys.modules:
            m = types.ModuleType(stub)
            sys.modules[stub] = m
    sys.modules["skimage"].transform = sys.modules["skimage.transform"]
    cuda_stub = types.ModuleType("pcdet.ops.roiaware_pool3d.roiaware_pool3d_cuda")
    sys.modules["pcdet.ops.roiaware_pool3d.roiaware_pool3d_cuda"] = cuda_stub
    sys.modules["pcdet.ops.roiaware_pool3d"].roiaware_pool3d_cuda = cuda_stub

    ns = types.SimpleNamespace()
    ns.common_utils = _load("pcdet.utils.common_utils", f"{P}/utils/common_utils.py")
    _load("pcdet.ops.roiaware_pool3d.roiaware_pool3d_utils", f"{P}/ops/roiaware_pool3d/roiaware_pool3d_utils.py")
    ns.box_utils = _load("pcdet.utils.box_utils", f"{P}/utils/box_utils.py")
    ns.data_processor = _load("pcdet.datasets.processor.data_processor",
                              f"{P}/datasets/processor/data_processor.py")
    ns.spconv_utils = _load("pcdet.utils.spconv_utils", f"{P}/utils/spconv_utils.py")
    _load("pcdet.models.backbones_3d.vfe.vfe_template", f"{P}/models/backbones_3d/vfe/vfe_template.py")
    ns.mean_vfe = _load("pcdet.models.backbones_3d.vfe.mean_vfe", f"{P}/models/backbones_3d/vfe/mean_vfe.py")
    ns.height_compression = _load("pcdet.models.backbones_2d.map_to_bev.height_compression",
                                  f"{P}/models/backbones_2d/map_to_bev/height_compression.py")
    ns.spconv_backbone = _load("pcdet.models.backbones_3d.spconv_backbone",
                               f"{P}/models/backbones_3d/spconv_backbone.py")
    ns.load_mixers = lambda: _load_mixers(ns, P)
    ns.DataProcessor = ns.data_processor.DataProcessor
    ns.MeanVFE = ns.mean_vfe.MeanVFE
    ns.HeightCompression = ns.height_compression.HeightCompression
    ns.VoxelBackBone8x = ns.spconv_backbone.VoxelBackBone8x
    ns.VoxelResBackBone8x = ns.spconv_backbone.VoxelResBackBone8x
    return ns


def _load_mixers(ns, P):
    """The reference's point mixers (SURVEY.md section 8 f-1), loaded on demand: they import the compiled iou3d_nms
    extension, which the point-level code paths exercised by the golden generator never call -- stubbed."""
    for name in ["pcdet.ops.iou3d_nms", "pcdet.datasets.augmentor"]:
        if name not in sys.modules:
            _pkg(name)
            parent, _, leaf = name.rpartition(".")
            setattr(sys.modules[parent], leaf, sys.modules[name])
    stub = types.ModuleType("pcdet.ops.iou3d_nms.iou3d_nms_utils")
    sys.modules["pcdet.ops.iou3d_nms.iou3d_nms_utils"] = stub
    sys.modules["pcdet.ops.iou3d_nms"].iou3d_nms_utils = stub
    try:      # pure numpy (get_points_in_box L474-491); imports only common_utils / box_utils, both loaded above
        ns.augmentor_utils = _load("pcdet.datasets.augmentor.augmentor_utils", f"{P}/datasets/augmentor/augmentor_utils.py")
    except Exception:
        aug = types.ModuleType("pcdet.datasets.augmentor.augmentor_utils")
        aug.get_points_in_box = None      # only used by the collision-detection variant, not exercised
        sys.modules["pcdet.datasets.augmentor.augmentor_utils"] = aug
        sys.modules["pcdet.datasets.augmentor"].augmentor_utils = aug
        ns.augmentor_utils = None
    ns.cutmix = _load("pcdet.datasets.processor.inter_domain_point_cutmix", f"{P}/datasets/processor/inter_domain_point_cutmix.py")
    ns.polarmix = _load("pcdet.datasets.processor.inter_domain_point_polarmix",
                        f"{P}/datasets/processor/inter_domain_point_polarmix.py")
    ns.mixup = _load("pcdet.datasets.processor.intra_domain_point_mixup", f"{P}/datasets/processor/intra_domain_point_mixup.py")
    return ns
