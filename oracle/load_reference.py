"""Import the UNMODIFIED reference `neuralop/layers/spectral_convolution.py` in this container.

TEST INFRASTRUCTURE ONLY -- used by the `oracle/make_golden*.py` generators to mint the stored vectors
under `tests/golden/`. Neither the tests nor the product package import this.

`neuralop/__init__.py` transitively needs h5py/zencfg/... (absent), so the parent packages are
pre-seeded as empty namespace modules and only the one file (plus its three siblings
`einsum_utils`, `base_spectral_conv`, `resample`, and `neuralop/utils.py`) is executed.
"""
import importlib
import os
import sys
import types

REF_ROOT = os.environ.get("NEURALOP_REFERENCE", "/root/reference")
_SHIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_shim")


def reference_available():
    return os.path.isfile(os.path.join(REF_ROOT, "neuralop", "layers", "spectral_convolution.py"))


def load_reference_spectral_conv():
    """Returns the reference module object (its `.SpectralConv` is the unmodified class)."""
    if not reference_available():
        raise FileNotFoundError(f"reference tree not found at {REF_ROOT}")
    if _SHIM not in sys.path:
        sys.path.insert(0, _SHIM)
    for name, path in [("neuralop", os.path.join(REF_ROOT, "neuralop")),
                       ("neuralop.layers", os.path.join(REF_ROOT, "neuralop", "layers"))]:
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.__path__ = [path]
            sys.modules[name] = m
    return importlib.import_module("neuralop.layers.spectral_convolution")
