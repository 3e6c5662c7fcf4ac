"""Import the UNMODIFIED reference modules from a checkout of the reference (REF_ROOT below).

FIXTURE GENERATION ONLY.  The reference is not part of this repository, so no test, smoke() or
bench.py may call this; oracle/make_golden.py uses it to write tests/golden/, which the tests
compare against.

Three shims are needed (SURVEY.md §8c):
  1. utils/util.py:6,10 import matplotlib.pyplot and skimage at module top (absent here);
  2. models/NonlocalNet.py:9 imports models/vgg19_gray.py which torch.load()s a missing
     checkpoint at import time (vgg19_gray.py:128);
  3. test.py is never imported (module-level torch.cuda.set_device(0), test.py:26).
"""
import os
import sys
import types

REF_ROOT = os.environ.get("DVC_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isfile(os.path.join(REF_ROOT, "models", "NonlocalNet.py"))


def load():
    """Returns a namespace with WarpNet, VGG19_pytorch, ColorVidNet, frame_colorization, util helpers."""
    if not available():
        raise RuntimeError("reference tree not present at " + REF_ROOT)
    saved_models = {k: v for k, v in sys.modules.items() if k == "models" or k.startswith("models.")}
    for k in saved_models:
        del sys.modules[k]
    for n in ["matplotlib", "matplotlib.pyplot", "skimage", "skimage.color", "skimage.io"]:
        if n not in sys.modules:
            sys.modules[n] = types.ModuleType(n)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["skimage"].color = sys.modules["skimage.color"]
    sys.modules["skimage"].io = sys.modules["skimage.io"]
    stub = types.ModuleType("models.vgg19_gray")
    stub.vgg19_gray = stub.vgg19_gray_new = object
    sys.modules["models.vgg19_gray"] = stub
    # the reference's `models/` has no __init__.py (namespace package); a regular `models` package
    # anywhere on sys.path (the drop-in's) would shadow it, so hide those entries during the import
    saved_path = list(sys.path)
    sys.path[:] = [REF_ROOT] + [q for q in saved_path if not os.path.isfile(os.path.join(q or ".", "models", "__init__.py"))]
    try:
        import contextlib
        import io

        with contextlib.redirect_stdout(io.StringIO()):
            from models.NonlocalNet import WarpNet, VGG19_pytorch
            from models.ColorVidNet import ColorVidNet
            from models.FrameColor import frame_colorization
            from utils.util import tensor_lab2rgb, uncenter_l, feature_normalize, gray2rgb_batch
            try:  # training-side consumer of the dense contraction (SURVEY.md §8f row 4); needs torchvision at import
                from models.ContextualLoss import ContextualLoss_forward
            except Exception:  # pragma: no cover
                ContextualLoss_forward = None
        ns = types.SimpleNamespace(
            WarpNet=WarpNet, VGG19_pytorch=VGG19_pytorch, ColorVidNet=ColorVidNet,
            frame_colorization=frame_colorization, tensor_lab2rgb=tensor_lab2rgb, uncenter_l=uncenter_l,
            feature_normalize=feature_normalize, gray2rgb_batch=gray2rgb_batch, ContextualLoss_forward=ContextualLoss_forward,
        )
    finally:
        sys.path[:] = saved_path
        # leave no `models.*` / `utils.*` entries of the reference behind: the drop-in package uses
        # the same module names
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.") or k == "utils"
                  or k.startswith("utils.") or k == "lib" or k.startswith("lib.")]:
            del sys.modules[k]
        sys.modules.update(saved_models)
    return ns


def build_modules(ns, sds, dtype=None):
    """Instantiate the reference nn.Modules and load our seeded state_dicts into them."""
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        warp, color, vgg = ns.WarpNet(1), ns.ColorVidNet(7), ns.VGG19_pytorch()
    warp.load_state_dict(sds["warp"])
    color.load_state_dict(sds["color"])
    vgg.load_state_dict(sds["vgg"])
    mods = [m.eval() for m in (vgg, warp, color)]
    if dtype is not None:
        mods = [m.to(dtype) for m in mods]
    for m in mods:
        for p in m.parameters():
            p.requires_grad = False
    return mods
