"""Parity of the CUDA path (through the C ABI, via the drop-in class) against the CPU oracle.

Bar (BASELINE.json north_star): masks bit-exact, warped RGB / depth within 1e-4 abs, normals within
0.01 degrees.  The kernels restate the reference's fp32 roundings, so these tests additionally assert
the stronger property that holds today: ZERO differing bits in every output.
"""
import numpy as np
import pytest
import torch

from tests import common as C

pytestmark = pytest.mark.gpu

RGBD_ATOL = 1e-4       # north_star: warped RGB and depth within 1e-4 absolute in fp32
NORMAL_ATOL_DEG = 0.01  # north_star: normals within 0.01 degrees


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _mk(cam_name, dev):
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    from oracle import oracle as O
    fx, fy, cx, cy = C.CAMERAS[cam_name]
    return Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy), O.Oracle(fx, fy, cx, cy)


def _check_params(w, o, I_g, I_a, dev):
    H, R, Hi = w._build_homography(_t(I_g, dev), _t(I_a, dev))
    oH, oR, oHi = o.build_homography(I_g, I_a)
    assert C.count_bit_mismatches(R.cpu().numpy(), oR) == 0
    assert C.count_bit_mismatches(H.cpu().numpy(), oH) == 0
    assert C.count_bit_mismatches(Hi.cpu().numpy(), oHi) == 0
    prm = w.frame_params(_t(I_g, dev), _t(I_a, dev)).cpu().numpy()
    sc = o.frame_scale(oH)
    assert C.count_bit_mismatches(prm[:, 27:35], sc) == 0


@pytest.mark.parametrize("cam_name,B,roll,pitch", [("S1", 512, 30, 30), ("S2", 512, 30, 30), ("S3", 512, 75, 40),
                                                    ("default", 256, 89, 60), ("tiny", 256, 45, 45)])
def test_frame_params_bit_exact(cuda_device, oracle_mod, cam_name, B, roll, pitch):
    w, o = _mk(cam_name, cuda_device)
    I_g, I_a = C.random_gravity(B, seed=11, roll_deg=roll, pitch_deg=pitch)
    _check_params(w, o, I_g, I_a, cuda_device)


def test_frame_params_edge_cases(cuda_device, oracle_mod):
    for cam_name in ("S1", "S3"):
        w, o = _mk(cam_name, cuda_device)
        I_g, I_a = C.edge_case_gravity()
        _check_params(w, o, I_g, I_a, cuda_device)
        I_g, I_a = C.extreme_roll_gravity(64, seed=5)
        _check_params(w, o, I_g, I_a, cuda_device)


def _full_path(cam_name, B, I_g, I_a, dev, seed, sparse_depth=False, depth_mode="bilinear", smooth=False):
    w, o = _mk(cam_name, dev)
    Hh, Ww = int(w.H), int(w.W)
    rgb, depth, normals = C.random_images(B, Hh, Ww, seed, sparse_depth=sparse_depth)
    if smooth:
        rgb = C.smooth_images(B, Hh, Ww, seed)
    g, a = _t(I_g, dev), _t(I_a, dev)
    # --- reference-shaped calls (the drop-in API) ---
    H1, y = w.warp_with_gravity_center_aligned(_t(rgb, dev), g, a)
    H2, yd = w.warp_with_gravity_center_aligned(_t(depth, dev), g, a, interp_mode=depth_mode)
    H3, z = w.inverse_warp_normal_image_with_gravity_center_aligned(_t(normals, dev), g, a)
    zn = torch.nn.functional.normalize(z, dim=1)
    # --- fused entry points ---
    H4, rgb_w, depth_w, mask = w.warp_rgbd(_t(rgb, dev), _t(depth, dev), g, a, depth_mode=depth_mode)
    H5, nhat = w.unwarp_normals(_t(normals, dev), g, a)
    torch.cuda.synchronize()
    # --- oracle ---
    oH, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode=depth_mode)
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    from oracle import oracle as O
    ozn = O.normalize(oz)
    omask = O.validity_mask(oy)

    y, yd, z, zn = y.cpu().numpy(), yd.cpu().numpy(), z.cpu().numpy(), zn.cpu().numpy()
    rgb_w, depth_w, mask, nhat = rgb_w.cpu().numpy(), depth_w.cpu().numpy(), mask.cpu().numpy(), nhat.cpu().numpy()
    for Hx in (H1, H2, H3, H4, H5):
        assert C.count_bit_mismatches(Hx.cpu().numpy(), oH) == 0
    # tolerance bar of the north star
    assert np.nanmax(np.abs(y - oy)) <= RGBD_ATOL
    assert np.nanmax(np.abs(yd - oyd)) <= RGBD_ATOL
    err, ok = C.angular_error_deg(nhat, ozn)
    assert err.size == 0 or err.max() <= NORMAL_ATOL_DEG
    assert np.array_equal(nhat[:, 0][~ok] == 0, ozn[:, 0][~ok] == 0)
    assert np.array_equal(mask, omask)                         # masks bit-exact
    # the stronger property: identical bits everywhere
    assert C.count_bit_mismatches(y, oy) == 0
    assert C.count_bit_mismatches(yd, oyd) == 0
    assert C.count_bit_mismatches(z, oz) == 0
    assert C.count_bit_mismatches(nhat, ozn) == 0
    assert C.count_bit_mismatches(rgb_w, oy) == 0
    assert C.count_bit_mismatches(depth_w, oyd) == 0
    assert C.count_bit_mismatches(zn, ozn) <= zn.size // 1000   # torch's own normalize on GPU: informational
    return w, o


@pytest.mark.parametrize("cam_name,B,roll,pitch", [("tiny", 16, 45, 45), ("S1", 8, 30, 30), ("S2", 4, 30, 30), ("S3", 4, 75, 40)])
def test_warp_unwarp_matches_oracle(cuda_device, oracle_mod, cam_name, B, roll, pitch):
    I_g, I_a = C.random_gravity(B, seed=1234, roll_deg=roll, pitch_deg=pitch)
    _full_path(cam_name, B, I_g, I_a, cuda_device, seed=1)


def test_warp_unwarp_extreme_roll(cuda_device, oracle_mod):
    I_g, I_a = C.extreme_roll_gravity(7, seed=3)
    _full_path("S3", 7, I_g, I_a, cuda_device, seed=2)


def test_warp_unwarp_edge_cases(cuda_device, oracle_mod):
    I_g, I_a = C.edge_case_gravity()
    _full_path("S1", I_g.shape[0], I_g, I_a, cuda_device, seed=4)
    _full_path("tiny", I_g.shape[0], I_g, I_a, cuda_device, seed=4, smooth=True)


def test_sparse_depth_nearest_and_bilinear(cuda_device, oracle_mod):
    I_g, I_a = C.random_gravity(6, seed=77)
    _full_path("S1", 6, I_g, I_a, cuda_device, seed=5, sparse_depth=True, depth_mode="nearest")
    _full_path("S1", 6, I_g, I_a, cuda_device, seed=5, sparse_depth=True, depth_mode="bilinear")


def test_sampler_grids_match_oracle(cuda_device, oracle_mod):
    for cam_name in ("tiny", "S1"):
        w, o = _mk(cam_name, cuda_device)
        I_g, I_a = C.edge_case_gravity()
        Rt, grid, inv = w.image_sampler_forward_inverse(_t(I_g, cuda_device), _t(I_a, cuda_device))
        oRt, ogrid, oinv = o.image_sampler_forward_inverse(I_g, I_a)
        assert C.count_bit_mismatches(Rt.cpu().numpy(), oRt) == 0
        assert C.count_bit_mismatches(grid.cpu().numpy(), ogrid) == 0
        assert C.count_bit_mismatches(inv.cpu().numpy(), oinv) == 0


def test_input_size_differs_from_canvas(cuda_device, oracle_mod):
    """Forward warp of a 640x480 image into the 320x240 canvas (the demo path resizes; the API allows any size)."""
    w, o = _mk("S1", cuda_device)
    I_g, I_a = C.random_gravity(3, seed=9)
    rgb, _, _ = C.random_images(3, 480, 640, seed=6)
    _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), _t(I_g, cuda_device), _t(I_a, cuda_device))
    _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0


def test_channels_last_input_no_copy(cuda_device, oracle_mod):
    w, o = _mk("S1", cuda_device)
    I_g, I_a = C.random_gravity(4, seed=21)
    rgb, _, normals = C.random_images(4, int(w.H), int(w.W), seed=8)
    x = _t(rgb, cuda_device).contiguous(memory_format=torch.channels_last)
    _, y = w.warp_with_gravity_center_aligned(x, _t(I_g, cuda_device), _t(I_a, cuda_device))
    assert y.is_contiguous(memory_format=torch.channels_last)
    _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
    n = _t(normals, cuda_device).contiguous(memory_format=torch.channels_last)
    _, z = w.unwarp_normals(n, _t(I_g, cuda_device), _t(I_a, cuda_device), normalize=False)
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0


@pytest.mark.parametrize("cam_name,kind", [("S1", "random"), ("S2", "random"), ("S3", "roll"), ("azure489", "random"), ("tiny", "edge")])
def test_channels_last_fast_kernels(cuda_device, oracle_mod, cam_name, kind):
    """torch.channels_last three-channel images (a CNN that runs in that memory format) take their own sheared kernels
    (kernels_shear_cl.cuh: twelve loads off one address, a (96, 32) staging tile, one bulk tensor store): outputs come back
    channels-last and carry the bits of the planar path -- fused calls, both depth modes, coverage, and the reference-shaped
    methods; compile-time and run-time geometry, a canvas height that is not a multiple of the tile, extreme rolls."""
    cam = C.CAMERAS.get(cam_name) or (404.0, 404.0, 319.529, 244.1902)           # 640 x 489, the real Azure Kinect canvas
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    w = Warping2DOFAlignment(*cam)
    Hh, Ww = int(w.H), int(w.W)
    B = 5
    I_g, I_a = {"random": lambda: C.random_gravity(B, seed=99), "roll": lambda: C.extreme_roll_gravity(B, seed=4),
                "edge": lambda: C.edge_case_gravity()}[kind]()
    B = I_g.shape[0]
    rgb, depth, normals = C.random_images(B, Hh, Ww, seed=23)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    x, d, n = _t(rgb, cuda_device), _t(depth, cuda_device), _t(normals, cuda_device)
    xc, nc = x.contiguous(memory_format=torch.channels_last), n.contiguous(memory_format=torch.channels_last)
    is_cl = lambda t: t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()
    for mode in ("bilinear", "nearest"):
        H0, r0, d0, m0, c0 = w.warp_rgbd(x, d, g, a, depth_mode=mode, with_coverage=True)
        H1, r1, d1, m1, c1 = w.warp_rgbd(xc, d, g, a, depth_mode=mode, with_coverage=True)
        assert is_cl(r1) and torch.equal(r1, r0) and torch.equal(d1, d0) and torch.equal(m1, m0) and torch.equal(c1, c0) and torch.equal(H1, H0)
    _, r2, _, m2 = w.warp_rgbd(xc, None, g, a)
    assert is_cl(r2) and torch.equal(r2, r0) and torch.equal(m2, m0)
    _, y0 = w.warp_with_gravity_center_aligned(x, g, a)
    _, y1 = w.warp_with_gravity_center_aligned(xc, g, a)
    assert is_cl(y1) and torch.equal(y1, y0)
    for normalize in (True, False):
        _, z0 = w.unwarp_normals(n, g, a, normalize=normalize)
        _, z1 = w.unwarp_normals(nc, g, a, normalize=normalize)
        assert is_cl(z1) and torch.equal(z1, z0)
    _, z2 = w.inverse_warp_normal_image_with_gravity_center_aligned(nc, g, a)
    assert is_cl(z2) and torch.equal(z2, z0)
    p = w.prepare(g, a)
    assert torch.equal(w.warp_rgbd(xc, d, params=p)[1], w.warp_rgbd(x, d, g, a)[1])
    assert torch.equal(w.unwarp_normals(nc, params=p)[1], w.unwarp_normals(n, g, a)[1])


def test_outputs_a_tensor_map_cannot_describe(cuda_device, oracle_mod):
    """The TMA write-out needs 16-byte aligned outputs (and mask): a caller of the C ABI that hands over anything else gets the
    LSU write-out of the same kernels -- same bits, no error.  Outputs placed 4 / 8 bytes into their allocations."""
    import ctypes
    from vi_depth_completion_b200 import _cabi
    from vi_depth_completion_b200.warping_2dof_alignment import _image
    w, o = _mk("S1", cuda_device)
    B, Hh, Ww = 3, int(w.H), int(w.W)
    I_g, I_a = C.random_gravity(B, seed=77)
    rgb, depth, normals = C.random_images(B, Hh, Ww, seed=14)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    x, d, n = _t(rgb, cuda_device), _t(depth, cuda_device)[:, None].contiguous(), _t(normals, cuda_device)
    _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    _, od = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    stream = ctypes.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream)
    ws = w._params_ws(B, cuda_device)
    for off_f, off_m in ((1, 0), (2, 4), (0, 4), (0, 8)):                       # floats into the fp32 outputs, bytes into the mask
        buf_rgb = torch.zeros(B * 3 * Hh * Ww + 4, device=cuda_device); buf_dep = torch.zeros(B * Hh * Ww + 4, device=cuda_device)
        buf_z = torch.zeros(B * 3 * Hh * Ww + 4, device=cuda_device); buf_m = torch.zeros(B * Hh * Ww + 16, dtype=torch.uint8, device=cuda_device)
        y = buf_rgb[off_f:off_f + B * 3 * Hh * Ww].view(B, 3, Hh, Ww); yd = buf_dep[off_f:off_f + B * Hh * Ww].view(B, 1, Hh, Ww)
        z = buf_z[off_f:off_f + B * 3 * Hh * Ww].view(B, 3, Hh, Ww); m = buf_m[off_m:off_m + B * Hh * Ww].view(B, 1, Hh, Ww)
        xi, di, yi, ydi, ni, zi = _image(x), _image(d), _image(y), _image(yd), _image(n), _image(z)
        with torch.cuda.device(cuda_device):
            _cabi.check(_cabi.lib().vidc_warp_rgbd(ctypes.byref(w._cam), ctypes.byref(xi), ctypes.byref(di), g.data_ptr(), a.data_ptr(), B,
                                                   _cabi.VIDC_BILINEAR, ws.data_ptr(), None, ctypes.byref(yi), ctypes.byref(ydi),
                                                   m.data_ptr(), None, stream))
            _cabi.check(_cabi.lib().vidc_unwarp_normals(ctypes.byref(w._cam), ctypes.byref(ni), g.data_ptr(), a.data_ptr(), B, 0,
                                                        ws.data_ptr(), None, ctypes.byref(zi), None, stream))
        assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0, (off_f, off_m)
        assert C.count_bit_mismatches(yd.cpu().numpy()[:, 0], od) == 0, (off_f, off_m)
        assert np.array_equal(m.cpu().numpy(), oracle_mod.validity_mask(oy)), (off_f, off_m)
        assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0, (off_f, off_m)
        assert buf_m[:off_m].sum().item() == 0 and buf_m[off_m + B * Hh * Ww:].sum().item() == 0       # nothing written outside


def test_coverage_counts(cuda_device, oracle_mod):
    w, o = _mk("S1", cuda_device)
    I_g, I_a = C.random_gravity(5, seed=31)
    rgb, depth, _ = C.random_images(5, int(w.H), int(w.W), seed=9)
    _, rgb_w, _, mask, cov = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), _t(I_g, cuda_device), _t(I_a, cuda_device),
                                         with_coverage=True)
    assert np.array_equal(cov.cpu().numpy(), mask.cpu().numpy().reshape(5, -1).sum(1))


def test_feature_maps_with_more_than_four_channels(cuda_device, oracle_mod):
    """F.grid_sample takes any channel count: the drop-in warps a 7-channel map in plane groups (same frame parameters) and
    back-propagates through it, bit-identical to the oracle per channel / equal to the 3-channel gradients."""
    w, o = _mk("S1", cuda_device)
    B = 3
    I_g, I_a = C.random_gravity(B, seed=21)
    x = np.random.RandomState(4).rand(B, 7, 240, 320).astype(np.float32)
    g, a = torch.from_numpy(I_g).to(cuda_device), torch.from_numpy(I_a).to(cuda_device)
    for mode in ("bilinear", "nearest"):
        _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(x).to(cuda_device), g, a, interp_mode=mode)
        _, oy = o.warp_with_gravity_center_aligned(x, I_g, I_a, interp_mode=mode)
        assert y.shape == (B, 7, 240, 320) and C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
    xt = torch.from_numpy(x).to(cuda_device).requires_grad_(True)
    wt = torch.from_numpy(np.random.RandomState(5).randn(B, 7, 240, 320).astype(np.float32)).to(cuda_device)
    (w.warp_with_gravity_center_aligned(xt, g, a)[1] * wt).sum().backward()
    x3 = torch.from_numpy(x[:, 4:7].copy()).to(cuda_device).requires_grad_(True)
    (w.warp_with_gravity_center_aligned(x3, g, a)[1] * wt[:, 4:7]).sum().backward()
    assert torch.allclose(xt.grad[:, 4:7], x3.grad, rtol=0, atol=2e-5)     # atomics: rounding-level differences only


def test_alignment_batch_must_match(cuda_device):
    """ADVICE r1: a shorter I_a used to be read out of bounds.  The reference fails at I_a[i] (:41, IndexError) or at the
    batched product I_a @ I_g (:43, RuntimeError); so does the drop-in, before any kernel sees the pointers."""
    w, _ = _mk("S1", cuda_device)
    g = torch.zeros(4, 3, device=cuda_device); g[:, 1] = 1
    img = torch.zeros(4, 3, 240, 320, device=cuda_device)
    with pytest.raises(IndexError):
        w.warp_with_gravity_center_aligned(img, g, g[:1])
    with pytest.raises(RuntimeError):
        w.inverse_warp_normal_image_with_gravity_center_aligned(img, g[:2], g)      # I_a longer than I_g ... and x.shape[0] != B
    with pytest.raises(RuntimeError):
        w._build_homography(g[:3], g)
    with pytest.raises(RuntimeError):
        w.warp_rgbd(img, None, g.reshape(2, 6), g)


def test_errors(cuda_device):
    w, _ = _mk("S1", cuda_device)
    g = torch.zeros(2, 3, device=cuda_device); g[:, 1] = 1
    with pytest.raises(AssertionError):                     # reference :123
        w.warp_with_gravity_center_aligned(torch.zeros(3, 3, 240, 320, device=cuda_device), g, g)
    with pytest.raises(RuntimeError):
        w.warp_with_gravity_center_aligned(torch.zeros(2, 3, 240, 320, device=cuda_device, dtype=torch.float64), g, g)
    with pytest.raises(RuntimeError):
        w.warp_with_gravity_center_aligned(torch.zeros(2, 3, 240, 320), g, g)          # CPU tensor: no fallback
    with pytest.raises(RuntimeError):
        w.inverse_warp_normal_image_with_gravity_center_aligned(torch.zeros(2, 3, 100, 100, device=cuda_device), g, g)
    img = torch.zeros(2, 3, 240, 320, device=cuda_device)
    with pytest.raises(ValueError, match="expected mode to be"):        # F.grid_sample's own check (reference :150)
        w.warp_with_gravity_center_aligned(img, g, g, interp_mode="cubic")
    with pytest.raises(ValueError):
        w.warp_rgbd(img, img[:, 0], g, g, depth_mode="linear")
    with pytest.raises(NotImplementedError):                            # bicubic: reference-shaped forward methods only
        w.warp_rgbd(img, img[:, 0], g, g, depth_mode="bicubic")
    wt, _ = _mk("tiny", cuda_device)                                    # frames ride on gridDim.z: explicit limit
    big = torch.zeros(1, 3, 48, 64, device=cuda_device).expand(65536, 3, 48, 64)
    gb = g[:1].expand(65536, 3).contiguous()
    with pytest.raises(RuntimeError, match="65535"):
        wt.warp_with_gravity_center_aligned(big, gb, gb)
    x = torch.zeros(2, 3, 240, 320, device=cuda_device, requires_grad=True)
    _, y = w.unwarp_normals(x, g, g)                        # fused renormalising entry point: forward-only
    with pytest.raises(NotImplementedError):
        y.sum().backward()
    # the same for the fused forward entry (with and without coverage counts): never a silent zero gradient
    import warnings
    for kw in ({}, {"with_coverage": True}):
        x = torch.rand(2, 3, 240, 320, device=cuda_device, requires_grad=True)
        out = w.warp_rgbd(x, torch.rand(2, 240, 320, device=cuda_device), g, g, **kw)
        assert out[1].requires_grad
        with warnings.catch_warnings():
            warnings.simplefilter("error")                              # torch's "autograd kernel was not registered" warning included
            with pytest.raises(NotImplementedError):
                out[1].sum().backward()
    x = torch.rand(2, 3, 240, 320, device=cuda_device, requires_grad=True)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        _, y = w.warp_with_gravity_center_aligned(x, g, g)
        y.sum().backward()                                              # differentiable method: no fallback node in the graph
    assert x.grad is not None and torch.isfinite(x.grad).all()


def test_empty_batch(cuda_device):
    w, _ = _mk("S1", cuda_device)
    g = torch.zeros(0, 3, device=cuda_device)
    H, y = w.warp_with_gravity_center_aligned(torch.zeros(0, 3, 240, 320, device=cuda_device), g, g)
    assert y.shape == (0, 3, 240, 320) and H.shape == (0, 3, 3)


_VARIANT_CODE = r'''
import sys, numpy as np, torch
sys.path.insert(0, %r)
from tests import common as C
from tests import exact_reference as X
from oracle import oracle as O
from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
dev = torch.device("cuda", 0)
t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
for cam, (I_g, I_a) in (("S1", C.random_gravity(6, 1234)), ("S2", C.random_gravity(3, 77)), ("S3", C.extreme_roll_gravity(7, 3)),
                        ("S1", C.random_gravity(5, 9, roll_deg=70, pitch_deg=40)), ("tiny", C.edge_case_gravity()),
                        ("S1", C.edge_case_gravity())):
    w, o = Warping2DOFAlignment(*C.CAMERAS[cam]), O.Oracle(*C.CAMERAS[cam])
    B = I_g.shape[0]
    rgb, depth, _ = C.random_images(B, o.H, o.W, 5)
    for mode in ("bilinear", "nearest"):
        _, rgb_w, depth_w, mask, cov = w.warp_rgbd(t(rgb), t(depth), t(I_g), t(I_a), depth_mode=mode, with_coverage=True)
        _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
        _, od = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode=mode)
        om = O.validity_mask(oy)
        assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0, (cam, mode, "rgb")
        assert C.count_bit_mismatches(depth_w.cpu().numpy(), od) == 0, (cam, mode, "depth")
        assert np.array_equal(mask.cpu().numpy(), om), (cam, mode, "mask")
        assert np.array_equal(cov.cpu().numpy().astype(np.int64), om.reshape(B, -1).sum(1).astype(np.int64)), (cam, mode, "coverage")
        _, y3 = w.warp_with_gravity_center_aligned(t(rgb), t(I_g), t(I_a), interp_mode=mode)       # reference-shaped calls
        _, y1 = w.warp_with_gravity_center_aligned(t(depth), t(I_g), t(I_a), interp_mode=mode)     # 3-D depth path (:110-112)
        _, o3 = o.warp_with_gravity_center_aligned(rgb, I_g, I_a, interp_mode=mode)
        assert C.count_bit_mismatches(y3.cpu().numpy(), o3) == 0, (cam, mode, "warp_with_gravity_center_aligned rgb")
        assert y1.dim() == 3 and C.count_bit_mismatches(y1.cpu().numpy(), od) == 0, (cam, mode, "warp_with_gravity_center_aligned depth")
    _, rgb_only, _, mask_only = w.warp_rgbd(t(rgb), None, t(I_g), t(I_a))
    assert C.count_bit_mismatches(rgb_only.cpu().numpy(), oy) == 0 and np.array_equal(mask_only.cpu().numpy(), om), (cam, "rgb only")
    nrm = C.random_images(B, o.H, o.W, 6)[2]
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(t(nrm), t(I_g), t(I_a))
    _, nh, valid = w.unwarp_normals(t(nrm), t(I_g), t(I_a), with_valid=True)
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(nrm, I_g, I_a)
    assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0, (cam, "unwarp")
    assert C.count_bit_mismatches(nh.cpu().numpy(), O.normalize(oz)) == 0, (cam, "unwarp+normalize")
    assert np.array_equal(valid.cpu().numpy().reshape(-1), X.touch_plane(o, I_g, I_a).reshape(-1)), (cam, "valid flags")
# signed zeros / denormals / inf / NaN through the same variant
w, o = Warping2DOFAlignment(*C.CAMERAS["S1"]), O.Oracle(*C.CAMERAS["S1"])
rgb, depth, nrm = C.special_value_images(4, o.H, o.W, 21)
I_g, I_a = C.special_value_gravity(4)
with np.errstate(all="ignore"):
    _, rgb_w, depth_w, mask = w.warp_rgbd(t(rgb), t(depth), t(I_g), t(I_a))
    _, nh = w.unwarp_normals(t(nrm), t(I_g), t(I_a))
    _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
    _, od = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(nrm, I_g, I_a)
    assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0 and C.count_bit_mismatches(depth_w.cpu().numpy().reshape(od.shape), od) == 0
    assert np.array_equal(mask.cpu().numpy().reshape(-1), O.validity_mask(oy).reshape(-1))
    assert C.count_bit_mismatches(nh.cpu().numpy(), O.normalize(oz)) == 0
print("VARIANT_OK")
'''


@pytest.mark.parametrize("env", [{"VIDC_SHEAR": "0"}, {"VIDC_SHEAR": "1"}, {"VIDC_SHEAR": "2"}, {"VIDC_TMA": "1"},
                                 {"VIDC_TILE_SKIP": "0"}, {"VIDC_INV_BOX": "1"}, {"VIDC_TMA_STORE": "0"}],
                         ids=["straight-rows", "sheared-forward", "sheared-both", "tma-staged", "no-tile-skip", "inverse-box-staged", "lsu-write-out"])
def test_kernel_variants_match_oracle(cuda_device, oracle_mod, env):
    """Every kernel family behind the fused entry points, each selected by its environment switch in a fresh process:
    straight row segments (VIDC_SHEAR=0), sheared forward rows only (=1), sheared forward + inverse (=2, the default) and
    the opt-in TMA-staged kernels (VIDC_TMA=1); VIDC_TMA_STORE=0 replaces the default TMA write-out of the sheared kernels (bulk
    tensor stores from a planar staging tile) by their LSU write-out.  Same bits as the oracle for moderate, extreme (column-major tiles) and
    edge-case gravity, both depth modes, coverage counts, RGB-only calls, a canvas whose height is not a multiple of
    the tile (240) and the special-value images."""
    import os
    import subprocess
    import sys
    code = _VARIANT_CODE % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, **env), capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "VARIANT_OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]


def test_host_buffer_entry_point_pipelined(cuda_device, oracle_mod):
    """vidc_warp_unwarp_host (C ABI with HOST buffers, chunked H2D / kernels / D2H pipeline): ragged last chunk,
    pageable and pinned buffers, same bits as the oracle."""
    import ctypes
    from vi_depth_completion_b200 import _cabi
    w, o = _mk("S1", cuda_device)
    B = 37
    I_g, I_a = C.random_gravity(B, seed=5)
    rgb, depth, normals = C.random_images(B, o.H, o.W, seed=12)
    o_rgb, o_depth, o_mask, o_n = oracle_mod.warp_unwarp_mt(o, rgb, depth, normals, I_g, I_a, 4)
    for pinned in (False, True):
        mk = (lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()) if pinned else (lambda a: torch.from_numpy(np.ascontiguousarray(a)))
        h = [mk(x) for x in (rgb, depth, normals, I_g, I_a)]
        outs = [torch.zeros(B, 3, o.H, o.W), torch.zeros(B, o.H, o.W), torch.zeros(B, 1, o.H, o.W, dtype=torch.uint8), torch.zeros(B, 3, o.H, o.W)]
        if pinned:
            outs = [t.pin_memory() for t in outs]
        with torch.cuda.device(cuda_device):
            _cabi.check(_cabi.lib().vidc_warp_unwarp_host(ctypes.byref(w._cam), B, *[t.data_ptr() for t in h], *[t.data_ptr() for t in outs],
                                                          ctypes.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream)))
        assert C.count_bit_mismatches(outs[0].numpy(), o_rgb) == 0
        assert C.count_bit_mismatches(outs[1].numpy(), o_depth) == 0
        assert np.array_equal(outs[2].numpy(), o_mask)
        assert C.count_bit_mismatches(outs[3].numpy(), o_n) == 0
    assert _cabi.lib().vidc_release_workspace() == 0


def test_packed_rgbd_nhwc4_matches_oracle(cuda_device, oracle_mod):
    """Opt-in packed layout (channels-last, C = 4): one 128-bit load per tap; per-channel results identical."""
    for cam_name, (I_g, I_a) in (("S1", C.random_gravity(5, 91)), ("S3", C.extreme_roll_gravity(7, 3)), ("tiny", C.edge_case_gravity())):
        w, o = _mk(cam_name, cuda_device)
        B = I_g.shape[0]
        rgb, depth, _ = C.random_images(B, o.H, o.W, 13, sparse_depth=(cam_name == "S1"))
        x = torch.cat([_t(rgb, cuda_device), _t(depth, cuda_device)[:, None]], 1).contiguous(memory_format=torch.channels_last)
        for mode in ("bilinear", "nearest"):
            _, y, mask, cov = w.warp_rgbd_packed(x, _t(I_g, cuda_device), _t(I_a, cuda_device), depth_mode=mode, with_coverage=True)
            assert y.is_contiguous(memory_format=torch.channels_last)
            _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
            _, od = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode=mode)
            yn = y.cpu().numpy()
            assert C.count_bit_mismatches(yn[:, :3], oy) == 0
            assert C.count_bit_mismatches(yn[:, 3], od) == 0
            assert np.array_equal(mask.cpu().numpy(), oracle_mod.validity_mask(oy))
            assert np.array_equal(cov.cpu().numpy(), mask.cpu().numpy().reshape(B, -1).sum(1))


@pytest.mark.parametrize("intr", [(120.0, 118.0, 100.3, 70.2), (90.0, 95.0, 33.4, 47.9), (300.0, 300.0, 256.0, 128.0),
                                  (90.0, 95.0, 47.9, 24.7), (500.0, 500.0, 319.9, 244.3)])
def test_odd_canvas_sizes(cuda_device, oracle_mod, intr):
    """Canvas sizes that are not multiples of the 32x32 tile (201x141, 67x96: straight-row runtime-geometry kernels), widths
    that are (512x256, 96x50, 640x489 -- the real Azure Kinect canvas: sheared runtime-geometry kernels, the last two with
    a bottom tile row that overhangs), the generic-stride kernels, inputs of a different size than the canvas, strided views."""
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    fx, fy, cx, cy = intr
    w, o = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
    assert (int(w.W), int(w.H)) == (o.W, o.H)
    B = 5
    I_g, I_a = C.random_gravity(B, seed=8, roll_deg=80, pitch_deg=30)       # both shear orientations
    rgb, depth, normals = C.random_images(B, o.H, o.W, seed=3)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    _, rgb_w, depth_w, mask = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), g, a)
    _, nhat = w.unwarp_normals(_t(normals, cuda_device), g, a)
    o_rgb, o_depth, o_mask, o_n = oracle_mod.warp_unwarp_mt(o, rgb, depth, normals, I_g, I_a, 2)
    assert C.count_bit_mismatches(rgb_w.cpu().numpy(), o_rgb) == 0
    assert C.count_bit_mismatches(depth_w.cpu().numpy(), o_depth) == 0
    assert np.array_equal(mask.cpu().numpy(), o_mask)
    assert C.count_bit_mismatches(nhat.cpu().numpy(), o_n) == 0
    # a differently sized, non-contiguous input view (every second column of a wider buffer): generic-stride kernel
    wide = C.random_images(B, o.H + 7, 2 * (o.W + 5), seed=4)[0]
    view = _t(wide, cuda_device)[:, :, :, ::2]
    assert not view.is_contiguous()
    _, y = w.warp_with_gravity_center_aligned(view, g, a)
    _, oy = o.warp_with_gravity_center_aligned(np.ascontiguousarray(wide[:, :, :, ::2]), I_g, I_a)
    assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0


def test_cuda_graph_capture(cuda_device, oracle_mod):
    """The whole step is capturable in a CUDA graph (no host synchronisation, no allocation outside torch's pool):
    the launch-bound small-batch case replays as one graph launch and returns the same bits."""
    w, o = _mk("S1", cuda_device)
    B = 8
    I_g, I_a = C.random_gravity(B, seed=12)
    rgb, depth, normals = C.random_images(B, o.H, o.W, seed=9)
    x, d, n, g, a = (_t(v, cuda_device) for v in (rgb, depth, normals, I_g, I_a))
    w.warp_rgbd(x, d, g, a); w.unwarp_normals(n, g, a)          # warm the workspace caches outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        _, rgb_w, depth_w, mask = w.warp_rgbd(x, d, g, a)
        _, nhat = w.unwarp_normals(n, g, a)
    x.copy_(_t(C.random_images(B, o.H, o.W, seed=10)[0], cuda_device))      # new input, same buffers
    graph.replay()
    torch.cuda.synchronize()
    _, oy = o.warp_with_gravity_center_aligned(x.cpu().numpy(), I_g, I_a)
    _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
    assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0
    assert C.count_bit_mismatches(nhat.cpu().numpy(), oracle_mod.normalize(oz)) == 0


def test_forward_warp_of_normals_with_rotation(cuda_device, oracle_mod):
    """a7, warp_normal_image_with_gravity_center_aligned (:258-290).  The reference method raises at :259, so parity is
    against its evident intent: the forward warp of a4 (bit-exact, oracle) followed by z = R y (:288)."""
    w, o = _mk("S1", cuda_device)
    I_g, I_a = C.random_gravity(4, seed=41, roll_deg=50, pitch_deg=30)
    normals = C.random_images(4, o.H, o.W, seed=2)[2]
    for mode in ("bilinear", "nearest", "bicubic"):
        H, z = w.warp_normal_image_with_gravity_center_aligned(_t(normals, cuda_device), _t(I_g, cuda_device), _t(I_a, cuda_device), interp_mode=mode)
        oH, oy = o.warp_with_gravity_center_aligned(normals, I_g, I_a, interp_mode=mode)
        _, R, _ = o.build_homography(I_g, I_a)
        want = np.einsum("bck,bkhw->bchw", R.astype(np.float64), oy.astype(np.float64))
        assert C.count_bit_mismatches(H.cpu().numpy(), oH) == 0
        assert np.abs(z.cpu().numpy() - want).max() <= (2e-6 if mode != "bicubic" else 1e-5)   # bicubic overshoots: |values| up to ~6


def test_warp_with_explicit_homography(cuda_device, oracle_mod):
    """a8, warp_with_homography (:292-310): dead code in the reference (numpy @ CUDA tensor).  Parity against a numpy fp64
    restatement of those lines: bbox of the projected corners, NON-uniform kw / kh, inverse in fp64, grid, bilinear sample."""
    w, o = _mk("S1", cuda_device)
    W_, H_ = o.W, o.H
    I_g, I_a = C.random_gravity(3, seed=19, roll_deg=25, pitch_deg=20)
    Hm, _, _ = o.build_homography(I_g, I_a)
    x = C.smooth_images(3, H_, W_, seed=5)
    _, y = w.warp_with_homography(_t(x, cuda_device), torch.from_numpy(Hm))
    cx, cy = C.CAMERAS["S1"][2], C.CAMERAS["S1"][3]
    XX, YY = np.meshgrid(np.arange(W_, dtype=np.float64), np.arange(H_, dtype=np.float64))   # [row, col] layout directly
    corners = np.array([[0, 0, 1], [W_ - 1, 0, 1], [0, H_ - 1, 1], [W_ - 1, H_ - 1, 1]], np.float64).T
    for b in range(3):
        Hb = Hm[b].astype(np.float64)
        c = Hb @ corners; c /= c[2]
        kw = W_ / (c[0].max() - c[0].min()); kh = H_ / (c[1].max() - c[1].min())           # :299-300
        P = np.stack([XX / kw + c[0].min(), YY / kh + c[1].min(), np.ones_like(XX)]).reshape(3, -1)
        q = np.linalg.inv(Hb) @ P; q /= q[2]
        grid = np.stack([(q[0] - cx) / (W_ / 2), (q[1] - cy) / (H_ / 2)], -1).reshape(1, H_, W_, 2).astype(np.float32)
        want = o.grid_sample(x[b:b + 1], grid)
        assert np.abs(y[b:b + 1].cpu().numpy() - want).max() <= 1e-3



@pytest.mark.parametrize("cam_name", ["S1", "tiny", "S2"])
def test_special_values_match_oracle(cuda_device, oracle_mod, cam_name):
    """Signed zeros, denormals, huge values, inf and NaN (tests/common.py: special_value_images).  The fused kernels take
    reciprocal fast paths inside a magnitude window and IEEE sqrt / division outside it, pad with +0 taps and seed the
    R^T product from +0: every output must land on the oracle's bits (the oracle is pinned on the same inputs against
    the executed reference, tests/golden/golden_tiny_special.npz), at compile-time and runtime kernel geometries."""
    from oracle import oracle as O
    w, o = _mk(cam_name, cuda_device)
    B, Hh, Ww = 4, int(w.H), int(w.W)
    rgb, depth, normals = C.special_value_images(B, Hh, Ww, seed=21)
    I_g, I_a = C.special_value_gravity(B)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), g, a)
    _, ydn = w.warp_with_gravity_center_aligned(_t(depth, cuda_device), g, a, interp_mode="nearest")
    _, rgb_w, depth_w, mask = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), g, a)
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(_t(normals, cuda_device), g, a)
    _, nhat = w.unwarp_normals(_t(normals, cuda_device), g, a)
    from vi_depth_completion_b200 import normal_utils as NU
    nhat2 = NU.Normalize(z)                                        # vidc_normalize3 (contiguous, H*W % 4 == 0: vec4 kernel)
    with np.errstate(all="ignore"):
        _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
        _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
        _, oydn = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode="nearest")
        _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
        ozn = O.normalize(oz)
    assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
    assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0
    assert C.count_bit_mismatches(depth_w.cpu().numpy().reshape(oyd.shape), oyd) == 0
    assert C.count_bit_mismatches(ydn.cpu().numpy().reshape(oydn.shape), oydn) == 0
    assert np.array_equal(mask.cpu().numpy().reshape(-1), O.validity_mask(oy).reshape(-1))
    assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0
    assert C.count_bit_mismatches(nhat.cpu().numpy(), ozn) == 0
    assert C.count_bit_mismatches(nhat2.cpu().numpy(), ozn) == 0


def test_degenerate_gravity_matches_oracle(cuda_device, oracle_mod):
    """Zero / NaN / inf / overflowing gravity: parameters, grids and every output on the oracle's bits.  Non-finite
    sampling coordinates read as out of bounds (ATen's CUDA safe_downgrade_to_int_range, GridSampler.cuh:140-147): zeros."""
    from oracle import oracle as O
    for cam_name in ("tiny", "S1"):
        w, o = _mk(cam_name, cuda_device)
        I_g, I_a = C.degenerate_gravity()
        B, Hh, Ww = I_g.shape[0], int(w.H), int(w.W)
        g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
        with np.errstate(all="ignore"):
            _check_params(w, o, I_g, I_a, cuda_device)
            rgb, depth, normals = C.random_images(B, Hh, Ww, seed=3)
            Rt, grid, inv = w.image_sampler_forward_inverse(g, a)
            oRt, ogrid, oinv = o.image_sampler_forward_inverse(I_g, I_a)
            _, rgb_w, depth_w, mask = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), g, a)
            _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), g, a)
            _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(_t(normals, cuda_device), g, a)
            _, nhat = w.unwarp_normals(_t(normals, cuda_device), g, a)
            _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
            _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
            _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
            ozn = O.normalize(oz)
        assert C.count_bit_mismatches(Rt.cpu().numpy(), oRt) == 0
        assert C.count_bit_mismatches(grid.cpu().numpy(), ogrid) == 0
        assert C.count_bit_mismatches(inv.cpu().numpy(), oinv) == 0
        assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
        assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0
        assert C.count_bit_mismatches(depth_w.cpu().numpy().reshape(oyd.shape), oyd) == 0
        assert np.array_equal(mask.cpu().numpy().reshape(-1), O.validity_mask(oy).reshape(-1))
        assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0
        assert C.count_bit_mismatches(nhat.cpu().numpy(), ozn) == 0


def test_isolated_nonfinite_coordinate_inside_a_warp(cuda_device, oracle_mod):
    """A projective denominator that is exactly 0 at one pixel: that lane's coordinate is inf / NaN while the rest of its
    warp samples normally.  The pixel must come out 0 (out of bounds), not NaN from 0 * NaN weights."""
    from oracle import oracle as O
    w, o = _mk("S1", cuda_device)
    I_g, I_a = C.isolated_nonfinite_gravity()
    B, Hh, Ww = I_g.shape[0], int(w.H), int(w.W)
    with np.errstate(all="ignore"):
        _, ogrid, oinv = o.image_sampler_forward_inverse(I_g, I_a)
    assert 0 < (~np.isfinite(ogrid)).sum() + (~np.isfinite(oinv)).sum() < 64         # the cases are really in there
    rgb, depth, normals = C.random_images(B, Hh, Ww, seed=9)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    for env_ok in (True,):
        _, rgb_w, depth_w, mask = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), g, a)
        _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), g, a)
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(_t(normals, cuda_device), g, a)
        _, nhat = w.unwarp_normals(_t(normals, cuda_device), g, a)
    with np.errstate(all="ignore"):
        _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
        _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
        _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(normals, I_g, I_a)
        ozn = O.normalize(oz)
    assert not np.isnan(rgb_w.cpu().numpy()).any() and not np.isnan(z.cpu().numpy()).any()
    assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0
    assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
    assert C.count_bit_mismatches(depth_w.cpu().numpy().reshape(oyd.shape), oyd) == 0
    assert np.array_equal(mask.cpu().numpy().reshape(-1), O.validity_mask(oy).reshape(-1))
    assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0
    assert C.count_bit_mismatches(nhat.cpu().numpy(), ozn) == 0


def test_exterior_tile_bitmap_never_drops_a_pixel(cuda_device, oracle_mod):
    """The forward kernels skip 32x32 canvas tiles that frame_params_tiles_kernel marks as certainly outside the source
    footprint (a conservative corner test with a margin).  Many frames over the whole roll / pitch range, an all-ones and
    a random image: every output pixel on the oracle's bits, so no marked tile ever contained a pixel of the footprint."""
    from oracle import oracle as O
    for cam_name, B, roll, pitch, seed in (("S1", 192, 89, 75, 31), ("S1", 64, 30, 30, 32), ("S2", 24, 89, 75, 33)):
        w, o = _mk(cam_name, cuda_device)
        Hh, Ww = int(w.H), int(w.W)
        I_g, I_a = C.random_gravity(B, seed=seed, roll_deg=roll, pitch_deg=pitch)
        rs = np.random.RandomState(seed)
        I_a[B // 2:] = rs.randn(B - B // 2, 3).astype(np.float32)              # general alignment directions too
        rgb = np.ones((B, 3, Hh, Ww), np.float32)
        rgb[B // 3:] = C.random_images(B - B // 3, Hh, Ww, seed=seed)[0]
        depth = C.random_images(B, Hh, Ww, seed=seed + 1)[1]
        g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
        _, rgb_w, depth_w, mask, cov = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), g, a, with_coverage=True)
        _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), g, a)
        with np.errstate(all="ignore"):
            _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
            _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
        om = O.validity_mask(oy)
        assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0
        assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
        assert C.count_bit_mismatches(depth_w.cpu().numpy().reshape(oyd.shape), oyd) == 0
        assert np.array_equal(mask.cpu().numpy().reshape(-1), om.reshape(-1))
        assert np.array_equal(cov.cpu().numpy().astype(np.int64), om.reshape(B, -1).sum(1).astype(np.int64))


def test_random_cameras_match_oracle(cuda_device, oracle_mod):
    """Fuzz over intrinsics: random canvas sizes (every third one with a width that is a multiple of 32, which takes the
    runtime-geometry sheared kernels; the others take the straight-row runtime-geometry kernels) and moderate / extreme /
    arbitrary gravity.  Fused and reference-shaped calls on the oracle's bits."""
    from oracle import oracle as O
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    rs = np.random.RandomState(77)
    for case in range(18):
        fx = float(rs.uniform(40, 500)); fy = float(fx * rs.uniform(0.9, 1.1))
        cx = float(rs.uniform(20, 180)); cy = float(rs.uniform(15, 120))
        if case % 3 == 0:
            cx = 16.0 * int(rs.randint(2, 12)) - 0.3                          # W = ceil(2 cx) = 32 k
        w, o = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy), oracle_mod.Oracle(fx, fy, cx, cy)
        assert (int(w.W), int(w.H)) == (o.W, o.H)
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
        rgb, depth, nrm = C.random_images(B, o.H, o.W, rs.randint(1 << 30))
        g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
        _, rgb_w, depth_w, mask = w.warp_rgbd(_t(rgb, cuda_device), _t(depth, cuda_device), g, a)
        _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), g, a)
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(_t(nrm, cuda_device), g, a)
        _, nhat = w.unwarp_normals(_t(nrm, cuda_device), g, a)
        with np.errstate(all="ignore"):
            _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
            _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a)
            _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(nrm, I_g, I_a)
            ozn = O.normalize(oz)
        tag = (case, fx, fy, cx, cy, o.W, o.H)
        assert C.count_bit_mismatches(rgb_w.cpu().numpy(), oy) == 0, tag
        assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0, tag
        assert C.count_bit_mismatches(depth_w.cpu().numpy().reshape(oyd.shape), oyd) == 0, tag
        assert np.array_equal(mask.cpu().numpy().reshape(-1), O.validity_mask(oy).reshape(-1)), tag
        assert C.count_bit_mismatches(z.cpu().numpy(), oz) == 0, tag
        assert C.count_bit_mismatches(nhat.cpu().numpy(), ozn) == 0, tag


def test_bicubic_matches_oracle_and_golden(cuda_device, oracle_mod):
    """interp_mode='bicubic' (valid in F.grid_sample, never used by the reference's callers): the reference-shaped forward
    methods on the oracle's bits and on the golden frozen from the executed reference -- contiguous, channels-last and 3-D
    depth inputs, extreme roll, special values, degenerate gravity, and the rotated forward warp of normals."""
    import os
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_tiny_bicubic.npz"))
    w, o = _mk("tiny", cuda_device)
    rgb, depth, _ = C.random_images(gold["I_g"].shape[0], int(w.H), int(w.W), int(gold["seed"]))
    g, a = _t(gold["I_g"], cuda_device), _t(gold["I_a"], cuda_device)
    _, y = w.warp_with_gravity_center_aligned(_t(rgb, cuda_device), g, a, interp_mode="bicubic")
    _, yd = w.warp_with_gravity_center_aligned(_t(depth, cuda_device), g, a, interp_mode="bicubic")
    assert yd.dim() == 3
    assert C.count_bit_mismatches(y.cpu().numpy(), gold["y_rgb"]) == 0
    assert C.count_bit_mismatches(yd.cpu().numpy(), gold["y_depth"]) == 0
    w, o = _mk("S1", cuda_device)
    Hh, Ww = int(w.H), int(w.W)
    cases = [(C.random_gravity(6, 3, 60, 45), C.random_images(6, Hh, Ww, 5)[0]),
             (C.extreme_roll_gravity(7, 2), C.random_images(7, Hh, Ww, 6)[0]),
             (C.special_value_gravity(4), C.special_value_images(4, Hh, Ww, 21)[0]),
             (C.degenerate_gravity(), C.random_images(C.degenerate_gravity()[0].shape[0], Hh, Ww, 3)[0])]
    for (I_g, I_a), img in cases:
        g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
        with np.errstate(all="ignore"):
            _, oy = o.warp_with_gravity_center_aligned(img, I_g, I_a, interp_mode="bicubic")
        _, y = w.warp_with_gravity_center_aligned(_t(img, cuda_device), g, a, interp_mode="bicubic")
        assert C.count_bit_mismatches(y.cpu().numpy(), oy) == 0
        _, ycl = w.warp_with_gravity_center_aligned(_t(img, cuda_device).contiguous(memory_format=torch.channels_last), g, a,
                                                    interp_mode="bicubic")
        assert C.count_bit_mismatches(ycl.cpu().numpy(), oy) == 0
    x = _t(cases[0][1], cuda_device).requires_grad_(True)               # forward only
    _, y = w.warp_with_gravity_center_aligned(x, _t(cases[0][0][0], cuda_device), _t(cases[0][0][1], cuda_device), interp_mode="bicubic")
    with pytest.raises(NotImplementedError):
        y.sum().backward()
