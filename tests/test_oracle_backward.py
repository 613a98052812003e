"""CPU checks of tests/backward_oracle.py, the serial row-major restatement of the ordered backward (vidc_warp_backward_ordered).

The reference's own autograd (frozen in golden_tiny_backward.npz) adds in a vectorised order that depends on the host ISA, so
the comparison is to rounding (2e-5 absolute); the fixed order itself is pinned bit for bit against the CUDA kernel in
tests/test_gpu_backward_ordered.py."""
import os

import numpy as np

from tests import backward_oracle as BO
from tests import common as C

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _golden(oracle_mod):
    g = np.load(os.path.join(GOLD, "golden_tiny_backward.npz"))
    orc = oracle_mod.Oracle(*g["cam"])
    wt = np.random.RandomState(int(g["wt_seed"])).randn(6, 3, orc.H, orc.W).astype(np.float32)
    return g, orc, wt


def test_oracle_backward_matches_reference_autograd(oracle_mod):
    g, orc, wt = _golden(oracle_mod)
    I_g, I_a = g["I_g"], g["I_a"]
    got_rgb = BO.warp_backward(orc, wt, I_g, I_a)
    got_depth = BO.warp_backward(orc, wt[:, 0], I_g, I_a)
    got_inv = BO.warp_backward(orc, wt, I_g, I_a, inverse=True)
    for name, got in (("grad_forward_rgb", got_rgb), ("grad_forward_depth", got_depth), ("grad_inverse_normals", got_inv)):
        ref = g[name]
        assert got.shape == ref.shape, name
        assert np.abs(got.astype(np.float64) - ref).max() <= 2e-5, name
        assert np.count_nonzero(ref) > 0.3 * ref.size, name          # the frames really overlap the image


def test_oracle_backward_is_the_adjoint_of_the_warp(oracle_mod):
    """<warp(x), g> == <x, warp_backward(g)> to rounding, for both modes and for an input smaller than the canvas."""
    _, orc, _ = _golden(oracle_mod)
    I_g, I_a = C.random_gravity(3, seed=12, roll_deg=40, pitch_deg=30)
    rs = np.random.RandomState(3)
    gout = rs.randn(3, 2, orc.H, orc.W).astype(np.float32)
    for mode in ("bilinear", "nearest"):
        for hw in ((orc.H, orc.W), (30, 41)):
            x = rs.randn(3, 2, *hw).astype(np.float32)
            _, y = orc.warp_with_gravity_center_aligned(x, I_g, I_a, interp_mode=mode)
            gx = BO.warp_backward(orc, gout, I_g, I_a, in_hw=hw, interp_mode=mode)
            lhs = float((y.astype(np.float64) * gout).sum())
            rhs = float((x.astype(np.float64) * gx).sum())
            assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs)), (mode, hw, lhs, rhs)
    n = rs.randn(3, 3, orc.H, orc.W).astype(np.float32)
    g3 = rs.randn(3, 3, orc.H, orc.W).astype(np.float32)
    _, z = orc.inverse_warp_normal_image_with_gravity_center_aligned(n, I_g, I_a)
    gn = BO.warp_backward(orc, g3, I_g, I_a, inverse=True)
    lhs, rhs = float((z.astype(np.float64) * g3).sum()), float((n.astype(np.float64) * gn).sum())
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs))


def test_oracle_backward_order_is_row_major(oracle_mod):
    """The serial scatter adds each contribution in output row-major order: a plain numpy loop restates it bit for bit."""
    _, orc, _ = _golden(oracle_mod)
    I_g, I_a = C.random_gravity(1, seed=5, roll_deg=60, pitch_deg=20)
    gout = np.random.RandomState(8).randn(1, 1, orc.H, orc.W).astype(np.float32)
    got = BO.warp_backward(orc, gout, I_g, I_a)
    Hm, _, Hi = orc.build_homography(I_g, I_a)
    grid = np.empty((1, orc.H, orc.W, 2), np.float32)
    oracle_mod.lib().vidc_oracle_forward_grid(oracle_mod.ctypes.byref(orc.cam), oracle_mod._p(Hm), oracle_mod._p(Hi), 1,
                                              oracle_mod._p(grid))
    assert np.isfinite(grid).all()
    f = np.float32

    def unnormalize(g, size):       # fma(g + 1, size, -1) / 2: the fp64 product and difference are exact, one rounding to fp32
        return f(f(np.float64(f(g + f(1))) * size - 1.0) / f(2))

    out = np.zeros((orc.H, orc.W), np.float32)
    for Y in range(orc.H):
        for X in range(orc.W):
            ix, iy = unnormalize(grid[0, Y, X, 0], orc.W), unnormalize(grid[0, Y, X, 1], orc.H)
            x0, y0 = np.floor(ix), np.floor(iy)
            w = [(f(x0 + 1) - ix) * (f(y0 + 1) - iy), (ix - x0) * (f(y0 + 1) - iy), (f(x0 + 1) - ix) * (iy - y0), (ix - x0) * (iy - y0)]
            for t, (xx, yy) in enumerate(((x0, y0), (x0 + 1, y0), (x0, y0 + 1), (x0 + 1, y0 + 1))):
                if 0 <= xx < orc.W and 0 <= yy < orc.H:
                    out[int(yy), int(xx)] = f(out[int(yy), int(xx)] + f(f(w[t]) * gout[0, 0, Y, X]))
    assert C.count_bit_mismatches(got[0, 0], out) == 0
