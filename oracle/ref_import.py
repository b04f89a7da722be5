"""oracle/ref_import.py -- TEST INFRASTRUCTURE (see oracle/__init__.py).

Imports the reference's own Python modules from /root/reference (present only
in the build container, never on the GPU box) with empty stubs for its missing
third-party dependencies (SURVEY.md Appendix F).  Used by
  * oracle/build_ref_kernels.py   (expands + compiles the reference CUDA kernels)
  * tests/golden/make_golden*.py  (generate the committed golden fixtures the tests compare against).
Nothing here is copied from the reference; it is imported where it lies.
"""
import os
import sys
import types

REF = os.environ.get("FVFI_REFERENCE", "/root/reference")


def available():
    return os.path.isdir(os.path.join(REF, "src"))


def _stub(name, **kw):
    m = types.ModuleType(name)
    m.__dict__.update(kw)
    sys.modules[name] = m
    return m


def install_stubs(steerable_cls=None):
    """Stub skimage/matplotlib/cupy/steerable so the reference modules import."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    if "skimage" not in sys.modules:
        from oracle import lab as _lab
        sk = _stub("skimage")
        sk.io = _stub("skimage.io")
        sk.color = _stub("skimage.color", rgb2lab=_lab.rgb2lab, lab2rgb=_lab.lab2rgb)
    if "matplotlib" not in sys.modules:
        mp = _stub("matplotlib")
        mp.pyplot = _stub("matplotlib.pyplot")
    if "cupy" not in sys.modules:
        cp = _stub("cupy")
        cp.memoize = lambda **k: (lambda f: f)
    if steerable_cls is None:
        from oracle.steerable_shim import SCFpyr_PyTorch as steerable_cls
    st = _stub("steerable")
    st.utils = _stub("steerable.utils")
    st.SCFpyr_PyTorch = _stub("steerable.SCFpyr_PyTorch", SCFpyr_PyTorch=steerable_cls)


def ref_adacof_module():
    """The reference's src/adacof/cupy_module/adacof.py (only cupy_kernel() and the
    kernel strings are usable without cupy)."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    if "cupy" not in sys.modules:
        cp = _stub("cupy")
        cp.memoize = lambda **k: (lambda f: f)
    import importlib
    return importlib.import_module("src.adacof.cupy_module.adacof")
