"""The oracle against the LIVE executed reference (beyond the frozen goldens) and the restated library functions
against torch itself.  The tests that execute the reference need its sources (oracle/ref_loader.py) and are skipped
where they are absent; no frozen copy of their comparisons exists, because the reference could not be executed when
the golden set was last extended (tests/golden holds what was frozen from it)."""
import ctypes
import warnings

import numpy as np
import pytest

from tests import common as C
from oracle.ref_loader import reference_available

needs_reference = pytest.mark.skipif(not reference_available(), reason="reference checkout not present")


def test_cos_restatement_matches_torch_cos(oracle_mod):
    """torch.cos on CPU (MKL VML vmsCos HA) vs oracle_cosf_mkl_ha on a dense sweep of [0, 1.6].
    (Every float in the interval -- 1.07e9 values -- was checked once with stride 1: 0 mismatches.)"""
    import torch
    bits = np.arange(0, int(np.float32(1.6).view(np.uint32)) + 1, 13, dtype=np.uint32)
    x = bits.view(np.float32)
    out = np.empty_like(x)
    oracle_mod.lib().vidc_oracle_cosf_array(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(x.size), out.ctypes.data_as(ctypes.c_void_p))
    ref = torch.cos(torch.from_numpy(x)).numpy()
    assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
    t = torch.from_numpy(x[::200003].copy())       # the 0-dim path the reference takes (ref :48)
    z = torch.stack([torch.cos(t[i]) for i in range(t.numel())]).numpy()
    assert np.array_equal(z.view(np.uint32), ref[::200003].view(np.uint32))


@needs_reference
def test_params_match_live_reference_random(oracle_mod):
    import torch
    from oracle.ref_loader import load_reference_class
    warnings.filterwarnings("ignore")
    Wref = load_reference_class("cpu")
    for cam_name, roll, pitch in (("S1", 30, 30), ("S3", 89, 60), ("default", 45, 45)):
        fx, fy, cx, cy = C.CAMERAS[cam_name]
        w, o = Wref(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
        I_g, I_a = C.random_gravity(192, seed=2024, roll_deg=roll, pitch_deg=pitch)
        rs = np.random.RandomState(1)
        I_a[96:] = rs.randn(96, 3).astype(np.float32)
        H, R, Hi = w._build_homography(torch.from_numpy(I_g), torch.from_numpy(I_a))
        oH, oR, oHi = o.build_homography(I_g, I_a)
        assert C.count_bit_mismatches(R.numpy(), oR) == 0
        assert C.count_bit_mismatches(H.numpy(), oH) == 0
        assert C.count_bit_mismatches(Hi.numpy(), oHi) == 0


@needs_reference
def test_full_path_matches_live_reference(oracle_mod):
    import torch
    from oracle.ref_loader import load_reference_class
    warnings.filterwarnings("ignore")
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["S1"]
    w, o = Wref(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
    I_g, I_a = C.extreme_roll_gravity(7, seed=11)
    rgb, depth, normals = C.random_images(7, o.H, o.W, seed=21)
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
    _, yd = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a, interp_mode="nearest")
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(normals), g, a)
    zn = torch.nn.functional.normalize(z, dim=1)
    _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode="nearest")
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    assert C.count_bit_mismatches(y.numpy(), oy) == 0
    assert C.count_bit_mismatches(yd.numpy(), oyd) == 0
    assert C.count_bit_mismatches(z.numpy(), oz) == 0
    assert C.count_bit_mismatches(zn.numpy(), oracle_mod.normalize(oz)) == 0


def test_sin_restatement_matches_torch_sin(oracle_mod):
    """torch.sin on CPU (MKL VML vmsSin HA).  Every float in [-3.2, 3.2] was checked once with stride 1: 0 mismatches."""
    import torch
    bits = np.concatenate([np.arange(0, int(np.float32(3.2).view(np.uint32)) + 1, 17, dtype=np.uint32),
                           np.arange(0x80000000, 0x80000000 + int(np.float32(3.2).view(np.uint32)) + 1, 19, dtype=np.uint32)])
    x = bits.view(np.float32)
    out = np.empty_like(x)
    oracle_mod.lib().vidc_oracle_sinf_array(x.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(x.size), out.ctypes.data_as(ctypes.c_void_p))
    assert np.array_equal(out.view(np.uint32), torch.sin(torch.from_numpy(x)).numpy().view(np.uint32))


@needs_reference
def test_special_values_match_live_reference(oracle_mod):
    """Signed zeros, denormals, inf, NaN at 320x240 against the executed reference (the 64x48 case is frozen as a golden)."""
    import torch
    from oracle.ref_loader import load_reference_class
    warnings.filterwarnings("ignore")
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["S1"]
    w, o = Wref(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
    rgb, depth, normals = C.special_value_images(4, o.H, o.W, seed=21)
    I_g, I_a = C.special_value_gravity(4)
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    with np.errstate(all="ignore"):
        _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
        _, ydn = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a, interp_mode="nearest")
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(normals), g, a)
        zn = torch.nn.functional.normalize(z, dim=1)
        _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
        _, oydn = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode="nearest")
        _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
        ozn = oracle_mod.normalize(oz)
    assert C.count_bit_mismatches(y.numpy(), oy) == 0
    assert C.count_bit_mismatches(ydn.numpy().reshape(oydn.shape), oydn) == 0
    assert C.count_bit_mismatches(z.numpy(), oz) == 0
    assert C.count_bit_mismatches(zn.numpy(), ozn) == 0


@needs_reference
def test_degenerate_gravity_against_live_reference(oracle_mod):
    """Zero / NaN / inf / overflowing gravity.  Parameters and sampling grids equal the executed reference bit for bit.
    Outputs equal it wherever the frame's sampling coordinates are finite.  KNOWN, DOCUMENTED divergence (DESIGN.md): for a
    non-finite coordinate the CPU build of ATen returns NaN in bilinear mode (0 * NaN weights) while its CUDA build -- the
    reference's deployment device -- returns 0 (safe_downgrade_to_int_range, GridSampler.cuh:140-147); the oracle and the
    kernels follow the CUDA build."""
    import torch
    from oracle.ref_loader import load_reference_class
    warnings.filterwarnings("ignore")
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    w, o = Wref(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
    I_g, I_a = C.degenerate_gravity()
    B = I_g.shape[0]
    rgb, depth, normals = C.random_images(B, o.H, o.W, seed=3)
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    with np.errstate(all="ignore"):
        H, R, Hi = w._build_homography(g, a)
        Rt, grid, inv = w.image_sampler_forward_inverse(g, a)
        _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
        _, ydn = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a, interp_mode="nearest")
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(normals), g, a)
        oH, oR, oHi = o.build_homography(I_g, I_a)
        oRt, ogrid, oinv = o.image_sampler_forward_inverse(I_g, I_a)
        _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
        _, oydn = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode="nearest")
        _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    for got, want in ((R, oR), (H, oH), (Hi, oHi), (Rt, oRt), (grid, ogrid), (inv, oinv)):
        assert C.count_bit_mismatches(got.numpy(), want) == 0
    assert C.count_bit_mismatches(ydn.numpy().reshape(oydn.shape), oydn) == 0      # nearest: 0 on both builds
    fwd_finite = np.isfinite(ogrid).all(axis=(1, 2, 3))
    inv_finite = np.isfinite(oinv).all(axis=(1, 2, 3))
    assert 3 <= (~fwd_finite).sum() < B
    assert C.count_bit_mismatches(y.numpy()[fwd_finite], oy[fwd_finite]) == 0
    assert C.count_bit_mismatches(z.numpy()[inv_finite], oz[inv_finite]) == 0
    assert np.isnan(y.numpy()[~fwd_finite]).all() and (oy[~fwd_finite] == 0).all()  # the divergence, exactly as documented


@needs_reference
def test_random_cameras_against_live_reference(oracle_mod):
    """Fuzz: random intrinsics (canvas sizes 40..400), moderate / extreme / arbitrary / un-normalised gravity.  Parameters and
    sampler grids bit-equal; warped outputs bit-equal except at isolated pixels where the projective denominator is exactly 0
    (the documented CPU-vs-CUDA ATen divergence: reference NaN, oracle 0).  A 15-minute run of this loop (3,180 cameras,
    19,080 frames) found nothing else."""
    import torch
    from oracle.ref_loader import load_reference_class
    warnings.filterwarnings("ignore")
    Wref = load_reference_class("cpu")
    rs = np.random.RandomState(2025)
    poles = 0
    for case in range(48):
        fx = float(rs.uniform(30, 700)); fy = float(fx * rs.uniform(0.9, 1.1))
        cx = float(rs.uniform(20, 200)); cy = float(rs.uniform(15, 150))
        w, o = Wref(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
        B, kind = 4, case % 4
        if kind == 0:
            I_g, I_a = C.random_gravity(B, rs.randint(1 << 30), 30, 30)
        elif kind == 1:
            I_g, I_a = C.random_gravity(B, rs.randint(1 << 30), 89, 80)
        elif kind == 2:
            I_g, I_a = rs.randn(B, 3).astype(np.float32), rs.randn(B, 3).astype(np.float32)
        else:
            I_g, I_a = C.random_gravity(B, rs.randint(1 << 30), 60, 60)
            I_g = (I_g * rs.uniform(0.1, 10, (B, 1))).astype(np.float32)
        rgb, _, nrm = C.random_images(B, o.H, o.W, rs.randint(1 << 30))
        g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
        with np.errstate(all="ignore"):
            H, R, Hi = w._build_homography(g, a)
            Rt, grid, inv = w.image_sampler_forward_inverse(g, a)
            _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
            _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(nrm), g, a)
            oH, oR, oHi = o.build_homography(I_g, I_a)
            oRt, ogrid, oinv = o.image_sampler_forward_inverse(I_g, I_a)
            _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
            _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(nrm, I_g, I_a)
        for got, want in ((R, oR), (H, oH), (Hi, oHi), (Rt, oRt), (grid, ogrid), (inv, oinv)):
            assert C.count_bit_mismatches(got.numpy(), want) == 0, (case, fx, fy, cx, cy)
        for got, want in ((y.numpy(), oy), (z.numpy(), oz)):
            diff = (C.bits(got) != C.bits(want)) & ~(np.isnan(got) & np.isnan(want))
            pole = np.isnan(got) & (want == 0)                      # denominator exactly 0: CPU ATen NaN, CUDA ATen / oracle 0
            assert not (diff & ~pole).any(), (case, fx, fy, cx, cy)
            poles += int(pole.any(axis=1).sum())
    assert poles < 200                                              # isolated pixels (whole non-finite frames excluded above by kind)


@needs_reference
def test_bicubic_matches_live_reference(oracle_mod):
    """interp_mode='bicubic' at 320x240 against the executed reference, including special values and degenerate gravity
    (non-finite coordinates give NaN in both builds of ATen for this mode, so there is no divergence to carve out)."""
    import torch
    from oracle.ref_loader import load_reference_class
    warnings.filterwarnings("ignore")
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["S1"]
    w, o = Wref(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
    cases = [(C.random_gravity(6, 3, 60, 45), C.random_images(6, o.H, o.W, 5)[0]),
             (C.extreme_roll_gravity(7, 2), C.random_images(7, o.H, o.W, 6)[0]),
             (C.special_value_gravity(4), C.special_value_images(4, o.H, o.W, 21)[0]),
             (C.degenerate_gravity(), C.random_images(C.degenerate_gravity()[0].shape[0], o.H, o.W, 3)[0])]
    for (I_g, I_a), img in cases:
        with np.errstate(all="ignore"):
            _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(img), torch.from_numpy(I_g), torch.from_numpy(I_a),
                                                      interp_mode="bicubic")
            _, oy = o.warp_with_gravity_center_aligned(img, I_g, I_a, interp_mode="bicubic")
        assert C.count_bit_mismatches(y.numpy(), oy) == 0
