"""Drop-in contract at the model level (SURVEY.md §4(ii), §8b): with the reference tree importable, swap the
videoad_b200 classes into ``model.backbone`` (``patch_reference``) and build the reference's own ``Mymodel`` with
them — parameter names and shapes must equal those of the unpatched model, and the reference's substring-based
grad toggles (backbone.py:44-76) must act on the same parameters.  CPU only (construction and state_dict; the
forward needs a B200) and skipped where ``oracle.ref_loader`` finds no copy of the original project."""
import os
import sys
import types

import pytest
import torch

from oracle import ref_loader

REF = ref_loader.ref_root()
pytestmark = pytest.mark.skipif(REF is None, reason="reference sources not staged (baseline/_ref or VADC_REFERENCE_ROOT)")


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules.setdefault(name, m)
    return sys.modules[name]


def _import_backbone():
    """stub recipe of SURVEY.md §8(c): timm / mmcv / mmaction.utils / matplotlib / skimage are absent here"""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    ident = type("DropPath", (torch.nn.Identity,), {"__init__": lambda self, *a, **k: torch.nn.Identity.__init__(self)})
    _stub("timm"); _stub("timm.models")
    _stub("timm.models.layers", DropPath=ident, trunc_normal_=torch.nn.init.trunc_normal_)
    _stub("mmcv"); _stub("mmcv.runner", load_checkpoint=lambda *a, **k: None)
    _stub("mmaction"); _stub("mmaction.utils", get_root_logger=lambda *a, **k: __import__("logging").getLogger("ref"))
    for n in ("matplotlib", "matplotlib.pyplot", "skimage", "skimage.io", "skimage.transform", "skimage.color"):
        try:
            __import__(n)
        except Exception:
            _stub(n)
    import model.backbone as bb
    return bb


def _build(bb):
    args = types.SimpleNamespace(patch_size=(2, 4, 4), frame_num=8, img_size=224)
    try:
        return bb.Mymodel(args, ispredict=True, iscluster=True)
    except TypeError:
        return bb.Mymodel(args)


def test_mymodel_builds_with_the_dropin_heads_and_keeps_its_state_dict():
    try:
        bb = _import_backbone()
        torch.manual_seed(0)
        ref = _build(bb)
    except Exception as e:                                   # a reference import problem is not this repo's failure
        pytest.skip(f"reference Mymodel does not build here: {e!r}")
    want = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
    ref_cluster_cls = type(ref.cluster1)
    import videoad_b200 as V
    patched = V.patch_reference()
    assert "model.backbone.cluster" in patched and "model.backbone.space_cluster" in patched
    try:
        mine = _build(bb)
        assert isinstance(mine.cluster1, V.EuclidDistance_Assign_Module) and not isinstance(mine.cluster1, ref_cluster_cls)
        assert isinstance(mine.space_cluster, V.Space_EuclidDistance_Assign_Module)
        got = {k: tuple(v.shape) for k, v in mine.state_dict().items()}
        assert got == want                                   # names, order and shapes: checkpoints are interchangeable
        mine.load_state_dict(ref.state_dict())               # the reference's weights load into the drop-in model
        # the reference's own grad toggles find the same parameters by name
        mine.cluster_on(); mine.cluster_center_on()
        assert mine.cluster1.cluster_center.requires_grad and mine.space_cluster.cluster_center.requires_grad
        assert not mine.cluster1.identity_matrix.requires_grad
        assert mine.cluster1.assign_func.alpha == ref.cluster1.assign_func.alpha == 16.0
        assert mine.space_cluster.assign_func.alpha == ref.space_cluster.assign_func.alpha == 32.0
    finally:
        import importlib
        import model.cluster
        importlib.reload(model.cluster)                      # undo the patch for other tests in this process
        bb.cluster = model.cluster.EuclidDistance_Assign_Module
        bb.space_cluster = model.cluster.Space_EuclidDistance_Assign_Module
