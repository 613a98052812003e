"""The CPU oracle (oracle/warp_oracle.c) against the golden vectors frozen from the EXECUTED reference
(oracle/make_golden.py).  Everything must match bit for bit.  Runs without a GPU."""
import hashlib
import os

import numpy as np
import pytest

from tests import common as C

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    return np.load(os.path.join(GOLD, f"golden_{name}.npz"))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _oracle_outputs(O, g):
    fx, fy, cx, cy = [float(v) for v in g["cam"]]
    o = O.Oracle(fx, fy, cx, cy)
    I_g, I_a, seed = g["I_g"], g["I_a"], int(g["seed"])
    B = I_g.shape[0]
    rgb, depth, normals = C.random_images(B, o.H, o.W, seed)
    sdepth = C.random_images(B, o.H, o.W, seed, sparse_depth=True)[1]
    H, R, Hi = o.build_homography(I_g, I_a)
    Rt, grid, inv = o.image_sampler_forward_inverse(I_g, I_a)
    _, y = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    _, yd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
    _, ydn = o.warp_with_gravity_center_aligned(sdepth, I_g, I_a, interp_mode="nearest")
    _, z = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    zn = O.normalize(z)
    mask = O.validity_mask(y)
    out = {"K": o.K, "K_inv": o.K_inv, "Hm": H, "R": R, "Hinv": Hi, "Rt_guard": Rt, "grid": grid, "inv_grid": inv,
           "y_rgb": y, "y_depth": yd, "y_sdepth_nearest": ydn, "z": z, "zn": zn, "mask": mask}
    for i, s in enumerate(((60, 80), (30, 40), (15, 20), (8, 10))):
        out[f"pyr{i}"] = O.mask_nearest(mask, s)
    gt = O.normalize(C.random_images(B, o.H, o.W, seed + 1000)[2])
    st = O.normal_stats(gt, z, mask.astype(np.float32), normalize_prediction=True)
    out["stats"] = st
    return o, out


BIG = ["grid", "inv_grid", "y_rgb", "y_depth", "y_sdepth_nearest", "z", "zn", "mask", "pyr0", "pyr1", "pyr2", "pyr3"]
SMALL = ["K", "K_inv", "Hm", "R", "Hinv", "Rt_guard"]


def _same_bits(a, b):
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    if a.dtype == np.uint8 or b.dtype == np.uint8:
        return np.array_equal(a.astype(np.uint8), b.astype(np.uint8))
    return C.count_bit_mismatches(a, b) == 0


def _check_digest(v, g, k):
    """k kept by the golden as SHA-256 + sampled values: the samples bit for bit, then the hash of all of v."""
    if v.dtype != np.uint8:
        v = v.astype(np.float32)
    assert tuple(g[k + "_shape"]) == v.shape, k
    assert np.array_equal(v.reshape(-1)[g[k + "_idx"]].view(np.uint8), g[k + "_val"].view(np.uint8)), f"sampled values differ in {k}"
    assert _sha(v) == str(g[k + "_sha256"]), f"SHA-256 of {k} differs from the executed reference"


def test_oracle_matches_reference_tiny_full(oracle_mod):
    g = _load("tiny")
    o, out = _oracle_outputs(oracle_mod, g)
    assert (o.W, o.H) == (int(g["W"]), int(g["H"]))
    for k in SMALL + BIG:
        if k + "_sha256" in g.files:
            _check_digest(out[k], g, k)
            continue
        assert out[k].shape == g[k].shape or out[k].size == g[k].size, k
        assert _same_bits(out[k].reshape(g[k].shape), g[k]), f"oracle differs from the executed reference in {k}"
    # the guard (:178-187) must have fired for at least one edge-case frame and not for all
    ident = np.all(g["Rt_guard"] == np.eye(3, dtype=np.float32), axis=(1, 2))
    assert ident.any() and not ident.all()


@pytest.mark.parametrize("name", ["S1", "S2", "S3"])
def test_oracle_matches_reference_full_resolution_digests(oracle_mod, name):
    g = _load(name)
    _, out = _oracle_outputs(oracle_mod, g)
    for k in SMALL:
        assert _same_bits(out[k], g[k]), k
    for k in BIG:
        _check_digest(out[k], g, k)


@pytest.mark.parametrize("name", ["tiny", "S1"])
def test_oracle_loss_statistics(oracle_mod, name):
    """normal_utils.py:20-34 / :7-17.  Sums are order-dependent in torch: compare to 1e-5 relative."""
    g = _load(name)
    _, out = _oracle_outputs(oracle_mod, g)
    loss1, ang1, loss2, ang2, msum = g["stats"]
    st = out["stats"]
    assert st["num"] == msum
    assert st["angle_sum"] == pytest.approx(ang1, rel=1e-5)
    assert st["angle_sum"] == pytest.approx(ang2, rel=1e-5)
    assert st["loss"] == pytest.approx(loss1, rel=1e-5)


@pytest.mark.parametrize("rule", ["azure", "scannet"])
def test_oracle_gravity_conditioning_matches_reference(oracle_mod, rule):
    g = _load("gravity")
    Ig, Ia = oracle_mod.condition_gravity(g["raw"], rule)
    assert C.count_bit_mismatches(Ig, g[rule + "_g"]) == 0
    assert C.count_bit_mismatches(Ia, g[rule + "_a"]) == 0


def test_oracle_matches_reference_special_values(oracle_mod):
    """Signed zeros, denormals, huge values, inf, NaN (golden_tiny_special.npz, from the executed reference): the sign of a
    zero result (+0 padding taps in grid_sample, +0 GEMM accumulator in bmm) and NaN propagation in F.normalize."""
    g = _load("tiny_special")
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    o = oracle_mod.Oracle(fx, fy, cx, cy)
    B = int(g["B"])
    rgb, depth, normals = C.special_value_images(B, o.H, o.W, int(g["seed"]))
    I_g, I_a = C.special_value_gravity(B)
    assert np.array_equal(I_g, g["I_g"]) and np.array_equal(I_a, g["I_a"])
    with np.errstate(all="ignore"):
        _, y = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
        _, yd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
        _, ydn = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode="nearest")
        _, z = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
        zn = oracle_mod.normalize(z)
    assert C.count_bit_mismatches(y, g["y_rgb"]) == 0
    assert C.count_bit_mismatches(yd, g["y_depth"].reshape(yd.shape)) == 0
    assert C.count_bit_mismatches(ydn, g["y_depth_nearest"].reshape(ydn.shape)) == 0
    assert C.count_bit_mismatches(z, g["z"]) == 0
    assert C.count_bit_mismatches(zn, g["zn"]) == 0
    assert np.array_equal(oracle_mod.validity_mask(y), g["mask"].reshape(oracle_mod.validity_mask(y).shape))
    # the cases are really in there: negative zeros survive the forward warp, none survive the GEMM, NaNs reach the output
    assert (np.signbit(g["y_rgb"]) & (g["y_rgb"] == 0)).sum() > 100
    assert (np.signbit(g["z"]) & (g["z"] == 0)).sum() == 0
    assert np.isnan(g["zn"]).sum() > 100 and np.isnan(g["y_rgb"]).sum() > 10


def test_oracle_bicubic_matches_reference(oracle_mod):
    """interp_mode='bicubic' (golden_tiny_bicubic.npz from the executed reference): RGB and the 3-D depth path, bit for bit."""
    g = _load("tiny_bicubic")
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    o = oracle_mod.Oracle(fx, fy, cx, cy)
    I_g, I_a = g["I_g"], g["I_a"]
    rgb, depth, _ = C.random_images(I_g.shape[0], o.H, o.W, int(g["seed"]))
    with np.errstate(all="ignore"):
        _, y = o.warp_with_gravity_center_aligned(rgb, I_g, I_a, interp_mode="bicubic")
        _, yd = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode="bicubic")
    assert C.count_bit_mismatches(y, g["y_rgb"]) == 0
    assert C.count_bit_mismatches(yd, g["y_depth"].reshape(yd.shape)) == 0


def test_oracle_demo_config(oracle_mod):
    """BASELINE config 1 (golden_demo.npz): the eight demo frames' real gravity through the Demo loader's conditioning and the
    warper at the main.py:243 intrinsics, the rasterised klt tracks as sparse depth -- SHA-256 of every output."""
    g = _load("demo")
    Ig, Ia = oracle_mod.condition_gravity(g["raw_gravity"], "azure")
    assert C.count_bit_mismatches(Ig, g["I_g"]) == 0 and C.count_bit_mismatches(Ia, g["I_a"]) == 0
    fx, fy, cx, cy = C.CAMERAS["S1"]
    o = oracle_mod.Oracle(fx, fy, cx, cy)
    B = 8
    rgb = C.smooth_images(B, o.H, o.W, int(g["rgb_seed"]))
    normals = C.random_images(B, o.H, o.W, int(g["normals_seed"]))[2]
    # sparse depth rebuilt from the stored tracks (fp64 pixel arithmetic of dataset.py:496-510)
    depth = np.zeros((B, o.H, o.W), np.float32)
    for b in range(B):
        for i in range(int(g["counts"][b])):
            t = g["tracks"][b, i]
            col, row = int(g["fc"][0] * (t[1] / t[3]) + g["cc"][0]), int(g["fc"][1] * (t[2] / t[3]) + g["cc"][1])
            if 0 <= row < o.H and 0 <= col < o.W:
                depth[b, row, col] = t[3]
    assert _sha(depth.reshape(B, 1, o.H, o.W)) == str(g["depth_sha256"])
    H, y = o.warp_with_gravity_center_aligned(rgb, Ig, Ia)
    _, yd = o.warp_with_gravity_center_aligned(depth, Ig, Ia)
    _, ydn = o.warp_with_gravity_center_aligned(depth, Ig, Ia, interp_mode="nearest")
    _, z = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, Ig, Ia)
    assert C.count_bit_mismatches(H, g["Hm"]) == 0
    assert _sha(y) == str(g["y_rgb_sha256"])
    assert _sha(yd) == str(g["y_depth_sha256"])
    assert _sha(ydn) == str(g["y_depth_nearest_sha256"])
    assert _sha(oracle_mod.validity_mask(y).astype(np.uint8)) == str(g["mask_sha256"])
    assert _sha(oracle_mod.normalize(z)) == str(g["zn_sha256"])
