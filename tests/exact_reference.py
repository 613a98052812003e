"""Exact references for four outputs that no serial restatement pins bit for bit: the atomic image backward of the two
reference-shaped warps (vidc_warp_backward), the validity plane of the inverse warp, the rotated forward warp and the
explicit-homography warp.  Checker of tests/test_exact_reference.py (the references themselves, on the CPU) and of the GPU
tests test_gpu_atomic_backward.py, test_gpu_validity_plane.py and test_gpu_forward_exact.py.

The grids and R come from the CPU oracle (oracle/oracle.py), as in tests/backward_oracle.py; the fp32 arithmetic is
tests/harness/exact_reference.c, built with gcc into a temporary directory on first use (the repository tree is not written).
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "harness", "exact_reference.c")
F_NAN, F_PINF, F_NINF, F_SUBNORMAL = 1, 2, 4, 8
U = 2.0 ** -24                     # unit roundoff of fp32
FLT_MAX = float(np.finfo(np.float32).max)
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(SRC, "rb").read()
        path = os.path.join(tempfile.gettempdir(), f"vidc_exact_reference_{os.getuid()}_{hashlib.sha256(src).hexdigest()[:16]}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}.tmp"
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-o", tmp, SRC,
                            "-lm"], check=True)
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
        _lib.vidc_test_homography_grid.argtypes = [ctypes.c_int, ctypes.c_int] + [ctypes.c_float] * 4 + [ctypes.c_void_p] * 2 + [
            ctypes.c_int, ctypes.c_void_p]
    return _lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def grids(orc, I_g, I_a, inverse):
    """(grid (B,H,W,2), R (B,3,3)) of the warp as the kernels sample it: the oracle's grids without the aspect guard."""
    Hm, R, Hi = orc.build_homography(I_g, I_a)
    B = Hm.shape[0]
    grid = np.empty((B, orc.H, orc.W, 2), np.float32)
    if inverse:
        O.lib().vidc_oracle_inverse_grid(ctypes.byref(orc.cam), O._p(Hm), B, O._p(grid))
    else:
        O.lib().vidc_oracle_forward_grid(ctypes.byref(orc.cam), O._p(Hm), O._p(Hi), B, O._p(grid))
    return grid, R


def scatter_stats(orc, grad_out, I_g, I_a, in_hw=None, inverse=False, interp_mode="bilinear"):
    """Per element of the image gradient ((B,C,Hin,Win), or (B,Hin,Win) for a (B,H,W) grad_out): the terms the backward
    scatters into it.  Returns a dict of arrays: k (count), E (exact sum of the finite terms, fp64), A (sum of their
    magnitudes), flags (F_NAN / F_PINF / F_NINF: such a term; F_SUBNORMAL: a subnormal term, or a subnormal sum of the
    first two), pair ((+0 + t1) + t2 in fp32: the result in every order when k <= 2)."""
    assert interp_mode in ("bilinear", "nearest")
    grad_out = O._f32(grad_out)
    squeeze = grad_out.ndim == 3
    if squeeze:
        grad_out = np.ascontiguousarray(grad_out[:, None])
    B, C = grad_out.shape[:2]
    assert grad_out.shape[2:] == (orc.H, orc.W) and C <= 64
    Hin, Win = (orc.H, orc.W) if in_hw is None else (int(in_hw[0]), int(in_hw[1]))
    assert not inverse or (C == 3 and (Hin, Win) == (orc.H, orc.W))
    grid, R = grids(orc, I_g, I_a, inverse)
    shape = (B, C, Hin, Win)
    out = dict(k=np.empty(shape, np.int32), E=np.empty(shape, np.float64), A=np.empty(shape, np.float64),
               flags=np.empty(shape, np.uint8), pair=np.empty(shape, np.float32))
    lib().vidc_test_scatter_stats(_p(grad_out), B, C, orc.H, orc.W, _p(grid), _p(R) if inverse else None, Hin, Win,
                                  0 if interp_mode == "bilinear" else 1, *(_p(out[n]) for n in ("k", "E", "A", "flags", "pair")))
    return {n: v[:, 0] for n, v in out.items()} if squeeze else out


def gamma(n):
    n = np.asarray(n, np.float64)
    return n * U / (1.0 - n * U)


def check_atomic_sum(S, st, what=""):
    """Asserts that S (fp32, any summation order of the terms of `st` from +0) is what such a sum can be:
      k = 0: +0;  a NaN term, or both infinities: NaN;  only one sign of infinity: that infinity (NaN too if the finite
      terms can overflow the other way);  k <= 2 without subnormals: the order-free (+0 + t1) + t2, bit for bit;
      finite terms with A <= FLT_MAX (1 - gamma): |S - E| <= gamma_{k-1} A + k 2^-52 A + k 2^-126 (the last term allows
      for subnormal inputs or results flushed to zero); larger A can overflow in some orders: not NaN.
    Returns the largest |S - E| / (gamma_{k-1} A) over the elements whose order matters (k >= 3) and whose sum no flushed
    subnormal can move noticeably (no subnormal term, gamma_{k-1} A >= 2^-100); 0.0 if there is none."""
    S = np.ascontiguousarray(S, np.float32)
    k, E, A, fl, pair = st["k"], st["E"], st["A"], st["flags"], st["pair"]
    assert S.shape == k.shape, (what, S.shape, k.shape)
    bits = S.view(np.uint32)
    nan, pinf, ninf = (fl & F_NAN) != 0, (fl & F_PINF) != 0, (fl & F_NINF) != 0
    g = gamma(np.maximum(k - 1, 0))
    safe = A <= FLT_MAX * (1.0 - g)

    def fail(mask, rule):
        idx = np.argwhere(mask)
        i = tuple(idx[0])
        return (f"{what}: {len(idx)} elements break '{rule}', first {i}: S={S[i]!r} k={k[i]} E={E[i]!r} A={A[i]!r} "
                f"flags={fl[i]} pair={pair[i]!r}")

    m = (k == 0) & (bits != 0)
    assert not m.any(), fail(m, "no term: +0")
    m = (nan | (pinf & ninf)) & ~np.isnan(S)
    assert not m.any(), fail(m, "NaN term or both infinities: NaN")
    one_inf = ~nan & (pinf ^ ninf)
    m = one_inf & pinf & ~((S == np.inf) | (~safe & np.isnan(S)))
    assert not m.any(), fail(m, "+inf terms only: +inf")
    m = one_inf & ninf & ~((S == -np.inf) | (~safe & np.isnan(S)))
    assert not m.any(), fail(m, "-inf terms only: -inf")
    finite = ~(nan | pinf | ninf) & (k > 0)
    m = finite & (k <= 2) & ((fl & F_SUBNORMAL) == 0) & (bits != pair.view(np.uint32))
    assert not m.any(), fail(m, "one or two terms: (+0 + t1) + t2")
    chk = finite & safe
    with np.errstate(invalid="ignore", over="ignore"):
        err = np.abs(S.astype(np.float64) - E)
    bound = g * A + k * 2.0 ** -52 * A + k * 2.0 ** -126
    m = chk & ~(err <= bound)
    assert not m.any(), fail(m, "|S - E| <= gamma_{k-1} A + k 2^-52 A + k 2^-126")
    m = finite & ~safe & np.isnan(S)
    assert not m.any(), fail(m, "finite terms: not NaN")
    r = chk & (k >= 3) & ((fl & F_SUBNORMAL) == 0) & (g * A >= 2.0 ** -100)
    return float((err[r] / (g[r] * A[r])).max()) if r.any() else 0.0


def touch_plane(orc, I_g, I_a):
    """(B,H,W) uint8 validity plane of the inverse warp: 1 where a bilinear tap of the pixel lies inside the canvas."""
    grid, _ = grids(orc, I_g, I_a, True)
    B = grid.shape[0]
    out = np.empty((B, orc.H, orc.W), np.uint8)
    lib().vidc_test_touch_plane(_p(grid), B, orc.H, orc.W, _p(out))
    return out


def rotate(y, R):
    """z = R y per pixel, as the rotated forward warp computes it: k-ascending FMA chain from +0."""
    y, R = O._f32(y), O._f32(R)
    B, C, H, W = y.shape
    assert C == 3 and R.shape == (B, 3, 3)
    z = np.empty_like(y)
    lib().vidc_test_rotate(_p(y), B, H, W, _p(R), _p(z))
    return z


def homography_params(Hm, W, H):
    """frame_params_from_h_kernel's fp64 block in its operation order (no FMA), cast to fp32: Hinv (B,3,3) and
    sc (B,4) = px_min, py_min, ikw, ikh."""
    h = O._f32(Hm).reshape(-1, 9).astype(np.float64)
    B = h.shape[0]
    Wm, Hmm = float(W - 1), float(H - 1)
    xmin, xmax = np.full(B, 1e300), np.full(B, -1e300)
    ymin, ymax = np.full(B, 1e300), np.full(B, -1e300)
    with np.errstate(all="ignore"):
        for cx, cy in ((0.0, 0.0), (Wm, 0.0), (0.0, Hmm), (Wm, Hmm)):
            c2 = h[:, 6] * cx + h[:, 7] * cy + h[:, 8]
            x = (h[:, 0] * cx + h[:, 1] * cy + h[:, 2]) / c2
            y = (h[:, 3] * cx + h[:, 4] * cy + h[:, 5]) / c2
            xmin, xmax, ymin, ymax = np.fmin(xmin, x), np.fmax(xmax, x), np.fmin(ymin, y), np.fmax(ymax, y)
        kw, kh = float(W) / (xmax - xmin), float(H) / (ymax - ymin)
        a = [h[:, i] for i in range(9)]
        det = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6])
        idet = 1.0 / det
        inv = np.stack([(a[4] * a[8] - a[5] * a[7]) * idet, (a[2] * a[7] - a[1] * a[8]) * idet, (a[1] * a[5] - a[2] * a[4]) * idet,
                        (a[5] * a[6] - a[3] * a[8]) * idet, (a[0] * a[8] - a[2] * a[6]) * idet, (a[2] * a[3] - a[0] * a[5]) * idet,
                        (a[3] * a[7] - a[4] * a[6]) * idet, (a[1] * a[6] - a[0] * a[7]) * idet, (a[0] * a[4] - a[1] * a[3]) * idet], 1)
        sc = np.stack([xmin, ymin, 1.0 / kw, 1.0 / kh], 1)
    return inv.astype(np.float32).reshape(B, 3, 3), sc.astype(np.float32)


def homography_grid(cam, Hinv, sc):
    """(B,H,W,2) grid of warp_with_homography.  cam: the product's vidc_camera (W, H, cx, cy, inv_half_w, inv_half_h)."""
    Hinv, sc = O._f32(Hinv), O._f32(sc)
    B = Hinv.shape[0]
    grid = np.empty((B, int(cam.H), int(cam.W), 2), np.float32)
    lib().vidc_test_homography_grid(int(cam.W), int(cam.H), cam.cx, cam.cy, cam.inv_half_w, cam.inv_half_h, _p(Hinv), _p(sc), B,
                                    _p(grid))
    return grid


def warp_with_homography(orc, cam, x, Hm):
    """Expected bits of warp_with_homography(x, Hm): x (B,C,Hin,Win), Hm (B,3,3) (already broadcast to the batch)."""
    Hinv, sc = homography_params(Hm, int(cam.W), int(cam.H))
    return orc.grid_sample(x, homography_grid(cam, Hinv, sc), "bilinear")
