"""Serial restatement of the ordered backward (vidc_warp_backward_ordered): the checker of tests/test_oracle_backward.py and
tests/test_gpu_backward_ordered.py.

The grids and R come from the CPU oracle (oracle/oracle.py); the row-major scatter is tests/harness/backward_scatter.c, built
with gcc into a temporary directory on first use (the repository tree is not written).
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "harness", "backward_scatter.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read()
        path = os.path.join(tempfile.gettempdir(), f"vidc_backward_scatter_{os.getuid()}_{hashlib.sha256(src).hexdigest()[:16]}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-o", tmp, SRC,
                            "-lm"], check=True)
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


def warp_backward(orc, grad_out, I_g, I_a, in_hw=None, inverse=False, interp_mode="bilinear"):
    """Gradient of warp_with_gravity_center_aligned (inverse=False) or inverse_warp_normal_image_with_gravity_center_aligned
    (inverse=True) w.r.t. the sampled image, in the fixed order: orc is an oracle.Oracle; grad_out (B,C,H,W) or (B,H,W) at the
    canvas size; in_hw = (Hin, Win) of the forward warp's input (default: the canvas).  Returns (B,C,Hin,Win) or (B,Hin,Win)."""
    assert interp_mode in ("bilinear", "nearest")
    grad_out, I_g, I_a = O._f32(grad_out), O._f32(I_g), O._f32(I_a)
    squeeze = grad_out.ndim == 3
    if squeeze:
        grad_out = np.ascontiguousarray(grad_out[:, None])
    B, C = grad_out.shape[:2]
    assert B == I_g.shape[0] and grad_out.shape[2:] == (orc.H, orc.W) and C <= 64
    Hin, Win = (orc.H, orc.W) if in_hw is None else (int(in_hw[0]), int(in_hw[1]))
    Hm, R, Hi = orc.build_homography(I_g, I_a)
    grid = np.empty((B, orc.H, orc.W, 2), np.float32)
    if inverse:
        assert C == 3 and (Hin, Win) == (orc.H, orc.W)
        O.lib().vidc_oracle_inverse_grid(ctypes.byref(orc.cam), O._p(Hm), B, O._p(grid))
    else:
        O.lib().vidc_oracle_forward_grid(ctypes.byref(orc.cam), O._p(Hm), O._p(Hi), B, O._p(grid))
    out = np.empty((B, C, Hin, Win), np.float32)
    lib().vidc_test_backward_scatter(O._p(grad_out), B, C, orc.H, orc.W, O._p(grid), O._p(R) if inverse else None, Hin, Win,
                                     0 if interp_mode == "bilinear" else 1, O._p(out))
    return out[:, 0] if squeeze else out
