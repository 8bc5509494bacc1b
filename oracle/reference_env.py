"""Import environment for the UNMODIFIED reference (git-ignored oracle/_ref, shipped by oracle/ship_reference.py
during build()).  TEST / BENCH INFRASTRUCTURE ONLY -- nothing under
`disentangling-vae_b200/` imports this.

Two kinds of shim, neither touching arithmetic (SURVEY.md section 8c, Appendix C):
  * stubs for modules that are absent from this image and unused on the path: `imageio`
    (disvae/training.py:1, utils/visualize.py:4 -- only `mimsave` at visualize.py:429) and `skimage.io`
    (utils/datasets.py:9 -- only used by the CelebA/Chairs downloaders);
  * `np.product = np.prod` (encoders.py:63, decoders.py:55 call the alias NumPy 2 removed).
"""
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CANDIDATES = [os.path.join(ROOT, "oracle", "_ref")]


def find_reference():
    for d in CANDIDATES:
        if os.path.isfile(os.path.join(d, "disvae", "training.py")) and os.path.isfile(os.path.join(d, "main.py")):
            return d
    return None


def install_stubs():
    import numpy as np
    if not hasattr(np, "product"):
        np.product = np.prod
    if "imageio" not in sys.modules:
        try:
            import imageio  # noqa: F401
        except ImportError:
            io = types.ModuleType("imageio")
            io.mimsave = lambda *a, **k: None
            io.mimread = lambda *a, **k: []
            sys.modules["imageio"] = io
    if "skimage" not in sys.modules:
        try:
            import skimage.io  # noqa: F401
        except ImportError:
            sk, skio = types.ModuleType("skimage"), types.ModuleType("skimage.io")
            skio.imread = lambda p: None
            sk.io = skio
            sys.modules.update({"skimage": sk, "skimage.io": skio})


def activate(ref_dir=None, package_first=None):
    """Put the reference on sys.path.  `package_first` = a directory holding another `disvae` package that must win
    the import (this repository's package, to drive it with the reference's main.py); None = the reference's own
    `disvae` is the one imported.  Returns the reference directory."""
    ref_dir = ref_dir or find_reference()
    if ref_dir is None:
        raise RuntimeError("reference not found (expected oracle/_ref: run oracle/ship_reference.py, or build(), "
                           "where a checkout of the reference is available)")
    sys.dont_write_bytecode = True
    install_stubs()
    for d in (ref_dir, package_first):
        if d is None:
            continue
        while d in sys.path:
            sys.path.remove(d)
        sys.path.insert(0, d)
    return ref_dir
