"""CPU checks of tests/exact_reference.py, the exact references of the atomic image backward, the validity plane, the rotated
forward warp and the explicit-homography warp: each reference is held against an independent statement of what it claims."""
import numpy as np
import pytest

from tests import backward_oracle as BO
from tests import common as C
from tests import exact_reference as X


def _unnormalize(g, size):
    """fmaf(g + 1, size, -1) / 2 in fp64: (g + 1) size - 1 is exact there (24 + 13 significant bits), one rounding to fp32."""
    gp1 = (g.astype(np.float32) + np.float32(1)).astype(np.float64)
    return (gp1 * size - 1.0).astype(np.float32) / np.float32(2)


def _safe(ix):
    with np.errstate(invalid="ignore"):
        return np.where(np.isfinite(ix) & (ix <= 2147483646.0) & (ix >= -2147483648.0), ix, np.float32(-100)).astype(np.float32)


def _in_bounds_taps(grid, Hin, Win, mode):
    """Per output pixel, the number of its taps inside the input (bilinear 0..4, nearest 0..1)."""
    ix, iy = _safe(_unnormalize(grid[..., 0], Win)), _safe(_unnormalize(grid[..., 1], Hin))
    if mode == "nearest":
        xn, yn = np.rint(ix), np.rint(iy)
        return ((xn >= 0) & (xn < Win) & (yn >= 0) & (yn < Hin)).astype(np.int64)
    x0, y0 = np.floor(ix).astype(np.int64), np.floor(iy).astype(np.int64)
    nx = ((x0 >= 0) & (x0 < Win)).astype(np.int64) + ((x0 + 1 >= 0) & (x0 + 1 < Win))
    ny = ((y0 >= 0) & (y0 < Hin)).astype(np.int64) + ((y0 + 1 >= 0) & (y0 + 1 < Hin))
    return nx * ny


def exact_edge_gravity():
    """Steep frames of the "tiny" canvas (64x48) on which some inverse-warp coordinates land exactly on -1 (a tap in bounds
    with weight 0) or on W-1 / H-1 (found by search)."""
    picks = ((131, 9), (143, 10), (3, 10), (146, 3))
    g = np.stack([C.random_gravity(16, seed=s, roll_deg=180, pitch_deg=85)[0][b] for s, b in picks])
    return g, np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (len(picks), 1))


def _cases():
    g_e, a_e = C.edge_case_gravity()
    g_r, a_r = C.random_gravity(4, seed=4242, roll_deg=70, pitch_deg=40)
    g_d, a_d = C.degenerate_gravity()
    g_s, a_s = C.special_value_gravity(4)
    yield "tiny", np.concatenate([g_e, g_r]), np.concatenate([a_e, a_r]), "random", None
    yield "tiny", g_d, a_d, "random", None
    yield "tiny", g_s, a_s, "special", None
    yield "S1", *C.random_gravity(2, seed=7, roll_deg=50, pitch_deg=30), "random", (7, 9)
    yield "S1", *C.random_gravity(2, seed=8, roll_deg=50, pitch_deg=30), "random", (121, 107)


def _grad(kind, B, Cc, H, W, seed):
    if kind == "special":
        rgb, _, normals = C.special_value_images(B, H, W, seed)
        return normals if Cc == 3 else rgb[:, :Cc]
    return np.random.RandomState(seed).randn(B, Cc, H, W).astype(np.float32)


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_serial_scatter_is_one_order_of_the_terms(oracle_mod, mode):
    """The serial scatter of backward_oracle is one valid summation order: it satisfies the bound of every element, equals
    (+0 + t1) + t2 wherever there are at most two terms, and the terms counted are the in-bounds taps times C."""
    for n, (cam, I_g, I_a, kind, in_hw) in enumerate(_cases()):
        orc = oracle_mod.Oracle(*C.CAMERAS[cam])
        for inverse in ((False, True) if in_hw is None else (False,)):
            Cc = 3 if (inverse or kind == "special") else 2
            gout = _grad(kind, I_g.shape[0], Cc, orc.H, orc.W, 30 + n)
            with np.errstate(all="ignore"):
                st = X.scatter_stats(orc, gout, I_g, I_a, in_hw=in_hw, inverse=inverse, interp_mode=mode)
                serial = BO.warp_backward(orc, gout, I_g, I_a, in_hw=in_hw, inverse=inverse, interp_mode=mode)
            what = f"{cam} {kind} in_hw={in_hw} inverse={inverse} {mode}"
            ratio = X.check_atomic_sum(serial, st, what)
            assert 0.0 <= ratio <= 1.0, what
            few = (st["k"] <= 2) & ((st["flags"] & (X.F_NAN | X.F_PINF | X.F_NINF)) == 0)
            assert C.count_bit_mismatches(serial[few], st["pair"][few]) == 0, what
            grid, _ = X.grids(orc, I_g, I_a, inverse)
            Hin, Win = (orc.H, orc.W) if in_hw is None else in_hw
            assert int(st["k"].sum()) == int(_in_bounds_taps(grid, Hin, Win, mode).sum()) * Cc, what


def test_bound_rejects_a_wrong_sum(oracle_mod):
    """The check is not vacuous: one ulp off an element with two or more terms, a lost term, or -0 where nothing landed,
    each fail it."""
    orc = oracle_mod.Oracle(*C.CAMERAS["tiny"])
    I_g, I_a = C.random_gravity(2, seed=3, roll_deg=40, pitch_deg=20)
    gout = np.random.RandomState(1).randn(2, 3, orc.H, orc.W).astype(np.float32)
    st = X.scatter_stats(orc, gout, I_g, I_a)
    good = BO.warp_backward(orc, gout, I_g, I_a)
    X.check_atomic_sum(good, st)
    i = tuple(np.argwhere((st["k"] == 2) & (good != 0))[0])
    bad = good.copy(); bad[i] = np.nextafter(bad[i], np.float32(np.inf))
    with pytest.raises(AssertionError):
        X.check_atomic_sum(bad, st)
    j = tuple(np.argwhere((st["k"] >= 4) & (np.abs(st["E"]) > 0.5))[0])
    bad = good.copy(); bad[j] = np.float32(st["E"][j] - st["A"][j] / st["k"][j])
    with pytest.raises(AssertionError):
        X.check_atomic_sum(bad, st)
    z = tuple(np.argwhere(st["k"] == 0)[0])
    bad = good.copy(); bad[z] = np.float32(-0.0)
    with pytest.raises(AssertionError):
        X.check_atomic_sum(bad, st)


def test_untouched_pixels_of_the_inverse_warp_are_plus_zero(oracle_mod):
    """Where no tap lies inside the canvas, the oracle's inverse warp is +0 in all three channels for any image when R is
    finite, and NaN in every channel that a non-finite entry of R reaches."""
    for cam, (I_g, I_a) in (("tiny", C.edge_case_gravity()), ("tiny", C.degenerate_gravity()), ("S1", C.isolated_nonfinite_gravity()),
                            ("S1", C.extreme_roll_gravity(7, 3))):
        orc = oracle_mod.Oracle(*C.CAMERAS[cam])
        B = I_g.shape[0]
        touch = X.touch_plane(orc, I_g, I_a)
        assert touch.any() or cam == "tiny"
        _, R, _ = orc.build_homography(I_g, I_a)
        for img in (C.random_images(B, orc.H, orc.W, 5)[2], np.concatenate([C.special_value_images(3, orc.H, orc.W, 6)[2]] * B)[:B]):
            with np.errstate(all="ignore"):
                _, z = orc.inverse_warp_normal_image_with_gravity_center_aligned(img, I_g, I_a)
            for b in range(B):
                off = touch[b] == 0
                for c in range(3):
                    col = R[b, :, c]
                    zc = z[b, c][off]
                    if np.isfinite(R[b]).all():
                        assert (C.bits(zc) == 0).all(), (cam, b, c)
                    elif not np.isfinite(col).all():
                        assert np.isnan(zc).all(), (cam, b, c)
        # a frame whose whole grid is non-finite touches nothing
        grid, _ = X.grids(orc, I_g, I_a, True)
        dead = ~np.isfinite(grid).any(axis=(1, 2, 3))
        assert not touch[dead].any()


def test_touch_plane_is_defined_by_tap_indices(oracle_mod):
    """touch is 1 exactly where the pixel's tap indices (x0|x0+1, y0|y0+1) meet the canvas, on frames steep enough that
    part of the camera image maps outside it; and a tap at exactly -1 is in bounds (weight 0) while one beyond is not."""
    orc = oracle_mod.Oracle(*C.CAMERAS["S1"])
    g_r, a_r = C.random_gravity(2, seed=17, roll_deg=60, pitch_deg=35)
    g_s, a_s = C.isolated_nonfinite_gravity()
    I_g, I_a = np.concatenate([g_r, g_s]), np.concatenate([a_r, a_s])
    touch = X.touch_plane(orc, I_g, I_a)
    grid, _ = X.grids(orc, I_g, I_a, True)
    want = _in_bounds_taps(grid, orc.H, orc.W, "bilinear") > 0
    assert np.array_equal(touch.astype(bool), want)
    assert 0 < touch.mean() < 1
    orc = oracle_mod.Oracle(*C.CAMERAS["tiny"])
    I_g, I_a = exact_edge_gravity()
    grid, _ = X.grids(orc, I_g, I_a, True)
    ix, iy = _unnormalize(grid[..., 0], orc.W), _unnormalize(grid[..., 1], orc.H)
    assert ((ix == -1) | (iy == -1)).any() and ((ix == orc.W - 1) | (iy == orc.H - 1)).any()
    touch = X.touch_plane(orc, I_g, I_a)
    assert touch[(ix == -1) & (iy > -1) & (iy < orc.H - 1)].all() and touch[(iy == -1) & (ix > -1) & (ix < orc.W - 1)].all()
    assert np.array_equal(touch.astype(bool), _in_bounds_taps(grid, orc.H, orc.W, "bilinear") > 0)


def test_rotation_with_identity_is_the_identity_but_for_signed_zero():
    rs = np.random.RandomState(2)
    y = rs.randn(3, 3, 5, 7).astype(np.float32)
    y[0, :, 0] = -0.0
    R = np.tile(np.eye(3, dtype=np.float32), (3, 1, 1))
    z = X.rotate(y, R)
    want = np.where(C.bits(y) == np.uint32(0x80000000), np.float32(0), y)
    assert C.count_bit_mismatches(z, want) == 0
    y[1, 1, 2] = np.inf                            # 0 * inf: an infinite component turns the others NaN
    y[2, 2, 3] = np.nan
    z = X.rotate(y, R)
    assert (z[1, 1, 2] == np.inf).all() and np.isnan(z[1, 0::2, 2]).all() and np.isnan(z[2, :, 3]).all()
    assert (C.bits(z[0, :, 0]) == 0).all()
    Rr = C.random_gravity(3, seed=1)[0]            # any matrix: the FMA chain, then compare with fp64
    Rm = np.stack([np.outer(v, v) + np.eye(3, dtype=np.float32) for v in Rr]).astype(np.float32)
    z = X.rotate(y[:, :, 1:2], Rm)
    ref = np.einsum("bck,bkhw->bchw", Rm.astype(np.float64), y[:, :, 1:2].astype(np.float64))
    ok = np.isfinite(ref)
    assert np.abs(z[ok] - ref[ok]).max() <= 4 * 2.0 ** -24 * np.abs(ref[ok]).max()


def test_homography_grid_matches_fp64_statement(oracle_mod):
    """The explicit-homography grid (fp32 chain over the fp64 parameter block) agrees with a plain fp64 restatement of the
    reference's lines (corners, bbox, non-uniform kw / kh, inverse, grid) to well below a thousandth of a pixel."""
    for cam, (I_g, I_a) in (("S1", C.random_gravity(3, seed=19, roll_deg=25, pitch_deg=20)), ("S2", C.extreme_roll_gravity(7, 5)),
                            ("tiny", C.random_gravity(3, seed=2, roll_deg=10, pitch_deg=70))):
        orc = oracle_mod.Oracle(*C.CAMERAS[cam])
        W_, H_ = orc.W, orc.H
        Hm, _, _ = orc.build_homography(I_g, I_a)
        Hinv, sc = X.homography_params(Hm, W_, H_)
        grid = X.homography_grid(orc.cam, Hinv, sc)
        cx, cy = C.CAMERAS[cam][2], C.CAMERAS[cam][3]
        XX, YY = np.meshgrid(np.arange(W_, dtype=np.float64), np.arange(H_, dtype=np.float64))
        corners = np.array([[0, 0, 1], [W_ - 1, 0, 1], [0, H_ - 1, 1], [W_ - 1, H_ - 1, 1]], np.float64).T
        for b in range(Hm.shape[0]):
            Hb = Hm[b].astype(np.float64)
            c = Hb @ corners; c /= c[2]
            kw = W_ / (c[0].max() - c[0].min()); kh = H_ / (c[1].max() - c[1].min())
            P = np.stack([XX / kw + c[0].min(), YY / kh + c[1].min(), np.ones_like(XX)]).reshape(3, -1)
            q = np.linalg.inv(Hb) @ P; q /= q[2]
            px = np.abs(grid[b, ..., 0].astype(np.float64).reshape(-1) * (W_ / 2) - (q[0] - cx))
            py = np.abs(grid[b, ..., 1].astype(np.float64).reshape(-1) * (H_ / 2) - (q[1] - cy))
            assert max(px.max(), py.max()) < 2e-4, (cam, b, px.max(), py.max())
