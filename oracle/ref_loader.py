"""TEST / BENCH INFRASTRUCTURE — imports the UNMODIFIED reference (a checkout of the original project named by the
environment variable ``VADC_REFERENCE_ROOT``, or the copy staged under ``baseline/_ref`` by scripts/stage_reference.py)
with the stub recipe of SURVEY.md 8(c).  Neither is part of this repository: without them the tests that build the
reference's own model skip.
Only tests/, ``__graft_entry__.smoke()`` and bench.py's reference legs may import this module; the product never does.

Stubs (packages the reference imports at module level but that are absent here and unused on the path):
``timm.models.layers`` {DropPath = identity (only instantiated when drop_path > 0, which the defaults never set:
swin_transformer.py:504), trunc_normal_}, ``mmcv.runner.load_checkpoint``, ``mmaction.utils.get_root_logger``,
``matplotlib``, ``skimage``."""
import logging
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CANDIDATES = tuple(c for c in (os.environ.get("VADC_REFERENCE_ROOT"), os.path.join(ROOT, "baseline", "_ref")) if c)


def ref_root():
    """directory holding the reference's ``model/cluster.py``, or None"""
    for c in CANDIDATES:
        if os.path.isfile(os.path.join(c, "model", "cluster.py")):
            return c
    return None


def _stub(name, **attrs):
    if name in sys.modules:
        m = sys.modules[name]
    else:
        m = types.ModuleType(name)
        sys.modules[name] = m
    for k, v in attrs.items():
        if not hasattr(m, k):
            setattr(m, k, v)
    return m


def install_stubs():
    class DropPath(torch.nn.Identity):
        def __init__(self, *a, **k):
            super().__init__()

    for name, attrs in (
        ("timm", {}), ("timm.models", {}),
        ("timm.models.layers", dict(DropPath=DropPath, trunc_normal_=torch.nn.init.trunc_normal_)),
        ("mmcv", {}), ("mmcv.runner", dict(load_checkpoint=lambda *a, **k: None)),
        ("mmaction", {}), ("mmaction.utils", dict(get_root_logger=lambda *a, **k: logging.getLogger("ref"))),
    ):
        try:
            __import__(name)
        except Exception:
            _stub(name, **attrs)
    for name in ("matplotlib", "matplotlib.pyplot", "skimage", "skimage.io", "skimage.transform", "skimage.color"):
        try:
            __import__(name)
        except Exception:
            _stub(name)
    sk = sys.modules["skimage"]
    for sub in ("io", "transform", "color"):
        if not hasattr(sk, sub):
            setattr(sk, sub, sys.modules["skimage." + sub])
    mp = sys.modules["matplotlib"]
    if not hasattr(mp, "pyplot"):
        mp.pyplot = sys.modules["matplotlib.pyplot"]


class Reference:
    """the reference's modules, imported once per process"""

    def __init__(self, root):
        self.root = root
        install_stubs()
        if root not in sys.path:
            sys.path.insert(0, root)
        from model import cluster, Memory
        from loss_tool import Recon_Loss
        self.cluster, self.Memory, self.Recon_Loss = cluster, Memory, Recon_Loss
        self._utils = self._backbone = None

    @property
    def utils(self):
        if self._utils is None:
            from misc import utils
            self._utils = utils
        return self._utils

    @property
    def backbone(self):
        if self._backbone is None:
            import model.backbone as bb
            self._backbone = bb
        return self._backbone

    def build_mymodel(self, patch_size=(2, 4, 4), ispredict=True, iscluster=True):
        """``Mymodel`` the way the live drivers build it (main_predict.py:164, contrast_evaluae.py:150)"""
        args = types.SimpleNamespace(patch_size=patch_size, frame_num=8, img_size=224)
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):          # the constructor prints one line per frozen parameter
            return self.backbone.Mymodel(args, ispredict=ispredict, iscluster=iscluster)


_ref = None


def load():
    """-> Reference, or None when neither $VADC_REFERENCE_ROOT nor baseline/_ref holds the reference"""
    global _ref
    if _ref is None:
        root = ref_root()
        if root is None:
            return None
        _ref = Reference(root)
    return _ref
