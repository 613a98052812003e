"""The CUDA path against the golden vectors frozen from the EXECUTED reference (tests/golden, made by
oracle/make_golden.py in the build container).  Bar: masks bit-exact, RGB / depth within 1e-4, normals within
0.01 degrees -- and, because the kernels restate the reference's roundings, identical bits / SHA-256."""
import hashlib
import os

import numpy as np
import pytest
import torch

from tests import common as C

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _cuda_outputs(g, dev):
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    from vi_depth_completion_b200 import normal_utils as NU
    fx, fy, cx, cy = [float(v) for v in g["cam"]]
    w = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy)
    I_g, I_a, seed = g["I_g"], g["I_a"], int(g["seed"])
    B = I_g.shape[0]
    Hh, Ww = int(w.H), int(w.W)
    rgb, depth, normals = C.random_images(B, Hh, Ww, seed)
    sdepth = C.random_images(B, Hh, Ww, seed, sparse_depth=True)[1]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    gg, aa = t(I_g), t(I_a)
    H, R, Hi = w._build_homography(gg, aa)
    Rt, grid, inv = w.image_sampler_forward_inverse(gg, aa)
    _, y = w.warp_with_gravity_center_aligned(t(rgb), gg, aa)
    _, yd = w.warp_with_gravity_center_aligned(t(depth), gg, aa)
    _, ydn = w.warp_with_gravity_center_aligned(t(sdepth), gg, aa, interp_mode="nearest")
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(t(normals), gg, aa)
    _, zn = w.unwarp_normals(t(normals), gg, aa, normalize=True)
    _, rgb_w, depth_w, mask = w.warp_rgbd(t(rgb), t(depth), gg, aa)
    maskf = NU.validity_mask(y)
    pyr = NU.pyramid_masks(maskf)
    pyr_from_u8 = NU.pyramid_masks(mask)                      # same levels straight from the fused kernel's uint8 mask
    assert all(torch.equal(p, q) for p, q in zip(pyr, pyr_from_u8))
    gt = torch.nn.functional.normalize(t(C.random_images(B, Hh, Ww, seed + 1000)[2]), dim=1)
    loss1, ang1 = NU.compute_normal_vectors_loss_l1(gt, z, maskf)
    loss2, ang2 = NU.compute_normal_vectors_loss_l2(gt, z, maskf)
    n = lambda x: x.detach().cpu().numpy()
    out = {"K": n(w.K), "K_inv": n(w.K_inv), "Hm": n(H), "R": n(R), "Hinv": n(Hi), "Rt_guard": n(Rt), "grid": n(grid),
           "inv_grid": n(inv), "y_rgb": n(y), "y_depth": n(yd), "y_sdepth_nearest": n(ydn), "z": n(z), "zn": n(zn),
           "mask": n(mask), "rgb_w": n(rgb_w), "depth_w": n(depth_w), "maskf": n(maskf).astype(np.uint8)}
    for i, p in enumerate(pyr):
        out[f"pyr{i}"] = n(p).astype(np.uint8)
    out["stats"] = [float(loss1), float(ang1), float(loss2), float(ang2), float(maskf.sum())]
    return out


def _check_digest(v, g, k):
    """k kept by the golden as SHA-256 + sampled values: the samples within 1e-4 and bit-equal, then the hash of all of v."""
    v = v.astype(np.uint8) if str(g[k + "_val"].dtype) == "uint8" else v.astype(np.float32)
    v = v.reshape(tuple(g[k + "_shape"]))
    got, want = v.reshape(-1)[g[k + "_idx"]], g[k + "_val"]
    if v.dtype == np.uint8:
        assert np.array_equal(got, want), k
    else:
        assert np.nanmax(np.abs(got - want)) <= 1e-4, k
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"sampled bits differ in {k}"
    assert _sha(v) == str(g[k + "_sha256"]), f"SHA-256 of {k} differs from the executed reference"


SMALL = ["K", "K_inv", "Hm", "R", "Hinv", "Rt_guard"]
BIG = ["grid", "inv_grid", "y_rgb", "y_depth", "y_sdepth_nearest", "z", "zn", "mask", "pyr0", "pyr1", "pyr2", "pyr3"]


def test_cuda_matches_reference_tiny_full(cuda_device):
    g = np.load(os.path.join(GOLD, "golden_tiny.npz"))
    out = _cuda_outputs(g, cuda_device)
    # north-star tolerances first
    assert np.array_equal(out["mask"].astype(np.uint8).reshape(g["mask"].shape), g["mask"])
    assert np.nanmax(np.abs(out["y_depth"] - g["y_depth"])) <= 1e-4
    err, ok = C.angular_error_deg(out["zn"], g["zn"])
    assert err.size == 0 or err.max() <= 0.01
    # and the stronger bit-level statement
    for k in SMALL + BIG:
        if k + "_sha256" in g.files:
            _check_digest(out[k], g, k)
            continue
        a, b = out[k], g[k]
        if b.dtype == np.uint8:
            assert np.array_equal(a.astype(np.uint8).reshape(b.shape), b), k
        else:
            assert C.count_bit_mismatches(a.reshape(b.shape), b) == 0, f"CUDA output differs from the executed reference in {k}"
    _check_digest(out["rgb_w"], g, "y_rgb")
    assert C.count_bit_mismatches(out["depth_w"].reshape(g["y_depth"].shape), g["y_depth"]) == 0
    assert np.array_equal(out["maskf"].reshape(g["mask"].shape), g["mask"])
    loss1, ang1, loss2, ang2, msum = g["stats"]
    s = out["stats"]
    assert s[4] == msum
    assert s[0] == pytest.approx(loss1, rel=1e-5) and s[1] == pytest.approx(ang1, rel=1e-5)
    assert s[2] == pytest.approx(loss2, rel=1e-5) and s[3] == pytest.approx(ang2, rel=1e-5)


@pytest.mark.parametrize("name", ["S1", "S2", "S3"])
def test_cuda_matches_reference_full_resolution_digests(cuda_device, name):
    g = np.load(os.path.join(GOLD, f"golden_{name}.npz"))
    out = _cuda_outputs(g, cuda_device)
    for k in SMALL:
        assert C.count_bit_mismatches(out[k], g[k]) == 0, k
    for k in BIG:
        _check_digest(out[k], g, k)


@pytest.mark.parametrize("rule", ["azure", "scannet"])
def test_cuda_gravity_conditioning_matches_reference(cuda_device, rule):
    """Row f1: raw IMU gravity -> (I_g, I_a) on device, bit-identical to the reference's dataset code."""
    from vi_depth_completion_b200.gravity import condition_gravity
    g = np.load(os.path.join(GOLD, "golden_gravity.npz"))
    Ig, Ia = condition_gravity(torch.from_numpy(g["raw"]).to(cuda_device), rule)
    assert C.count_bit_mismatches(Ig.cpu().numpy(), g[rule + "_g"]) == 0
    assert C.count_bit_mismatches(Ia.cpu().numpy(), g[rule + "_a"]) == 0


def test_cuda_backward_matches_reference_autograd(cuda_device):
    """Row f4: gradients w.r.t. the sampled image against torch autograd through the EXECUTED reference (CPU).
    The CUDA backward scatters with atomics, so the tolerance is rounding-level, not bit-exact: 2e-5 absolute on
    gradients of magnitude O(1..10)."""
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    g = np.load(os.path.join(GOLD, "golden_tiny_backward.npz"))
    fx, fy, cx, cy = [float(v) for v in g["cam"]]
    w = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy)
    I_g, I_a = g["I_g"], g["I_a"]
    B, Hh, Ww = I_g.shape[0], int(w.H), int(w.W)
    rgb, depth, normals = C.random_images(B, Hh, Ww, int(g["seed"]))
    wt = np.random.RandomState(int(g["wt_seed"])).randn(B, 3, Hh, Ww).astype(np.float32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    gg, aa, wtt = t(I_g), t(I_a), t(wt)
    x = t(rgb).requires_grad_(True)
    _, y = w.warp_with_gravity_center_aligned(x, gg, aa)
    (y * wtt).sum().backward()
    assert np.abs(x.grad.cpu().numpy() - g["grad_forward_rgb"]).max() <= 2e-5
    d = t(depth).requires_grad_(True)
    _, yd = w.warp_with_gravity_center_aligned(d, gg, aa)
    (yd * wtt[:, 0]).sum().backward()
    assert np.abs(d.grad.cpu().numpy() - g["grad_forward_depth"]).max() <= 2e-5
    n = t(normals).requires_grad_(True)
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(n, gg, aa)
    (z * wtt).sum().backward()
    assert np.abs(n.grad.cpu().numpy() - g["grad_inverse_normals"]).max() <= 2e-5
    n2 = t(normals).requires_grad_(True)
    _, z2 = w.inverse_warp_normal_image_with_gravity_center_aligned(n2, gg, aa)
    (torch.nn.functional.normalize(z2, dim=1) * wtt).sum().backward()      # torch's normalize backward on top of ours
    ref = g["grad_inverse_normals_normalized"]
    assert np.abs(n2.grad.cpu().numpy() - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())


def test_cuda_sparse_depth_rasterisation_matches_reference(cuda_device):
    """Row f2: point tracks -> (B,1,240,320) sparse depth on device, identical to the Demo loader's loop (dataset.py:496-510),
    including pixel collisions (last point wins), out-of-range points, empty frames and the eight demo_dataset track files;
    then warped (nearest, as is sensible for sparse samples) through the fused kernel."""
    from vi_depth_completion_b200.gravity import rasterize_sparse_depth
    g = np.load(os.path.join(GOLD, "golden_rasterize.npz"))
    tracks = torch.from_numpy(g["tracks"]).to(cuda_device)
    depth = rasterize_sparse_depth(tracks, g["counts"], g["fc"], g["cc"], 240, 320)
    assert depth.shape == (tracks.shape[0], 1, 240, 320)
    assert C.count_bit_mismatches(depth.cpu().numpy(), g["depth"]) == 0


def test_cuda_matches_reference_special_values(cuda_device):
    """golden_tiny_special.npz: the executed reference on signed zeros / denormals / huge / inf / NaN inputs."""
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    g = np.load(os.path.join(GOLD, "golden_tiny_special.npz"))
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    w = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy)
    B = int(g["B"])
    rgb, depth, normals = C.special_value_images(B, int(w.H), int(w.W), int(g["seed"]))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    gg, aa = t(g["I_g"]), t(g["I_a"])
    _, y = w.warp_with_gravity_center_aligned(t(rgb), gg, aa)
    _, yd = w.warp_with_gravity_center_aligned(t(depth), gg, aa)
    _, ydn = w.warp_with_gravity_center_aligned(t(depth), gg, aa, interp_mode="nearest")
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(t(normals), gg, aa)
    _, zn = w.unwarp_normals(t(normals), gg, aa, normalize=True)
    _, rgb_w, depth_w, mask = w.warp_rgbd(t(rgb), t(depth), gg, aa)
    for got, key in ((y, "y_rgb"), (rgb_w, "y_rgb"), (yd, "y_depth"), (depth_w, "y_depth"), (ydn, "y_depth_nearest"),
                     (z, "z"), (zn, "zn")):
        assert C.count_bit_mismatches(got.cpu().numpy().reshape(g[key].shape), g[key]) == 0, key
    assert np.array_equal(mask.cpu().numpy().reshape(-1), g["mask"].reshape(-1))


def test_cuda_demo_config_end_to_end(cuda_device):
    """BASELINE config 1 (golden_demo.npz): raw IMU gravity of the eight demo frames -> vidc_condition_gravity, their klt track
    files -> vidc_rasterize_sparse_depth, then the fused warp (bilinear and nearest depth) and unwarp at the main.py:243
    intrinsics: every stage on the bits the reference's loader code and warper produced."""
    from vi_depth_completion_b200.gravity import condition_gravity, rasterize_sparse_depth
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    g = np.load(os.path.join(GOLD, "golden_demo.npz"))
    fx, fy, cx, cy = C.CAMERAS["S1"]
    w = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy)
    Hh, Ww, B = int(w.H), int(w.W), 8
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    Ig, Ia = condition_gravity(t(g["raw_gravity"]), "azure")
    assert C.count_bit_mismatches(Ig.cpu().numpy(), g["I_g"]) == 0 and C.count_bit_mismatches(Ia.cpu().numpy(), g["I_a"]) == 0
    depth = rasterize_sparse_depth(t(g["tracks"]), g["counts"], g["fc"], g["cc"], Hh, Ww)
    assert _sha(depth.cpu().numpy()) == str(g["depth_sha256"])
    rgb = C.smooth_images(B, Hh, Ww, int(g["rgb_seed"]))
    normals = C.random_images(B, Hh, Ww, int(g["normals_seed"]))[2]
    H, rgb_w, depth_w, mask = w.warp_rgbd(t(rgb), depth, Ig, Ia)
    _, _, depth_n, _ = w.warp_rgbd(t(rgb), depth, Ig, Ia, depth_mode="nearest")
    _, zn = w.unwarp_normals(t(normals), Ig, Ia)
    assert C.count_bit_mismatches(H.cpu().numpy(), g["Hm"]) == 0
    assert _sha(rgb_w.cpu().numpy()) == str(g["y_rgb_sha256"])
    assert _sha(depth_w.cpu().numpy().reshape(B, Hh, Ww)) == str(g["y_depth_sha256"])
    assert _sha(depth_n.cpu().numpy().reshape(B, Hh, Ww)) == str(g["y_depth_nearest_sha256"])
    assert _sha(mask.cpu().numpy().reshape(B, 1, Hh, Ww)) == str(g["mask_sha256"])
    assert _sha(zn.cpu().numpy()) == str(g["zn_sha256"])
    assert abs(float(mask.float().mean()) - float(g["valid_fraction"])) < 1e-6
