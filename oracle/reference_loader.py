"""Make the UNMODIFIED reference importable in the authoring container.

TEST INFRASTRUCTURE (see oracle/prims.py header).  ``/root/reference`` exists only in the
authoring container, never on the GPU box: this module is used by
``tests/golden/make_golden.py`` to generate fixtures and by the optional
``tests/test_reference_live.py`` (skipped when the reference tree is absent).

What it does: puts ``oracle/shim`` (stand-ins for maskrcnn_benchmark / yacs / timm) and the
reference root on ``sys.path``, injects the two API-drift stubs the reference needs on a modern
stack (``np.int`` used at track_core.py:206; ``torchvision.models.utils`` imported at dla.py:11),
and returns the reference's own ``cfg`` and ``build_siammot``.
"""
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("SIAMMOT_REFERENCE_ROOT", "/root/reference")
_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "shim")
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "siammot", "modelling"))


def _patch_color_jitter():
    """Third API-drift stub: the reference pins torchvision 0.8 (requirements_exact.txt), whose ``ColorJitter.get_params``
    returned a callable transform; since 0.9 it returns (order, brightness, contrast, saturation, hue).  The reference's video
    transform calls the result (video_augmentation.py:98-105) -- also at test time, with all factors None.  Give it the
    callable back."""
    import torchvision.transforms as T
    import torchvision.transforms.functional as F
    if getattr(T.ColorJitter.get_params, "_drift_patched", False):
        return
    orig = T.ColorJitter.get_params

    def get_params(brightness, contrast, saturation, hue):
        r = orig(brightness, contrast, saturation, hue)
        if not isinstance(r, tuple):
            return r
        order, b, c, s, h = r

        def apply(img):
            for fn_id in order:
                if fn_id == 0 and b is not None:
                    img = F.adjust_brightness(img, b)
                elif fn_id == 1 and c is not None:
                    img = F.adjust_contrast(img, c)
                elif fn_id == 2 and s is not None:
                    img = F.adjust_saturation(img, s)
                elif fn_id == 3 and h is not None:
                    img = F.adjust_hue(img, h)
            return img
        return apply
    get_params._drift_patched = True
    T.ColorJitter.get_params = staticmethod(get_params)


def use_shim():
    """Put the repository and oracle/shim on sys.path: the stand-ins import without the reference tree."""
    for p in (_REPO, _SHIM):
        if p not in sys.path:
            sys.path.insert(0, p)


def load():
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    import numpy as np
    if not hasattr(np, "int"):
        np.int = int  # removed in numpy 1.24; track_core.py:206
    if "torchvision.models.utils" not in sys.modules:
        m = types.ModuleType("torchvision.models.utils")
        m.load_state_dict_from_url = lambda *a, **k: {}  # dla.py:403-405 (no network: random init)
        sys.modules["torchvision.models.utils"] = m
    _patch_color_jitter()
    for p in (_REPO, REFERENCE_ROOT, _SHIM):
        if p not in sys.path:
            sys.path.insert(0, p)
    from siammot.configs.defaults import cfg
    from siammot.modelling.rcnn import build_siammot
    return cfg, build_siammot
