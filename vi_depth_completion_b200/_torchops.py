"""Loader of the thin torch C++ extension (csrc/torch_ops.cpp -> _vidc_torch_ops.so): TORCH_LIBRARY operators `torch.ops.vidc.*`
in front of the C ABI.  The hot entry points of Warping2DOFAlignment reach libvidc_b200.so through these operators only (no
Python marshalling, traceable by torch.compile(fullgraph=True)); the ctypes binding (_cabi.py) carries the calls no operator
takes.  Like libvidc_b200.so, the extension is part of the product: ops() raises when it is missing or does not load.
"""
import os

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_vidc_torch_ops.so")
_ops = None


def ops():
    """torch.ops.vidc.  Raises RuntimeError (never falls back) when the extension has not been built or does not load."""
    global _ops
    if _ops is None:
        import torch
        from . import _cabi
        _cabi.lib()                                   # libvidc_b200.so first: a missing product library is the error shown
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: the torch extension is part of the product and there is no fallback. "
                               "Build it with `python -m vi_depth_completion_b200.build`.")
        try:
            torch.ops.load_library(LIB_PATH)
        except OSError as e:                          # e.g. built against another torch
            raise RuntimeError(f"{LIB_PATH} could not be loaded ({e}); rebuild it with "
                               "`python -m vi_depth_completion_b200.build --force`.") from None
        _ops = torch.ops.vidc
    return _ops
