"""Gradients with respect to I_g and I_a (vidc_warp_backward_params + vidc_frame_params_backward) on the B200, against the
torch restatement of the reference (tests/gravity_grad_reference.py): the fp64 restatement on smooth images, the fp32 one --
the reference as torch runs it -- on white noise.  The bar is a per-frame, norm-wise relative error of 1e-3."""
import warnings

import numpy as np
import pytest
import torch

from tests import common as C
from tests import gravity_grad_reference as GR

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
TOL = 1e-3


def _warper(cam_name):
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    return Warping2DOFAlignment(*C.CAMERAS[cam_name])


def _noise(shape, seed):
    return np.random.RandomState(seed).uniform(-1, 1, shape).astype(np.float32)


def _smooth(shape, seed):
    B, C_, H, W = shape
    rs = np.random.RandomState(seed)
    Y, X = np.meshgrid(np.arange(H) / H, np.arange(W) / W, indexing="ij")
    out = np.zeros(shape, np.float32)
    for b in range(B):
        for c in range(C_):
            f = rs.uniform(1.0, 3.0, 4)
            out[b, c] = np.sin(2 * np.pi * (f[0] * X + f[1] * Y) + f[2]) + 0.5 * np.cos(2 * np.pi * f[3] * X * Y)
    return out


def _ours(w, method, x, I_g, I_a, wt, wH, mode="bilinear"):
    g = torch.from_numpy(I_g).to(DEV).requires_grad_(True)
    a = torch.from_numpy(I_a).to(DEV).requires_grad_(True)
    if method == "homography":
        H, R, Hi = w._build_homography(g, a)
        L = (H * wt[0]).sum() + (R * wt[1]).sum() + (Hi * wt[2]).sum()
    else:
        if method == "warp":
            Hm, y = w.warp_with_gravity_center_aligned(x, g, a, interp_mode=mode)
        else:
            Hm, y = w.inverse_warp_normal_image_with_gravity_center_aligned(x, g, a)
        L = (y * wt).sum() + ((Hm * wH).sum() if wH is not None else 0.0)
    L.backward()
    return g.grad.double().cpu().numpy(), a.grad.double().cpu().numpy()


def _reference(w, method, x, I_g, I_a, wt, wH, dtype, mode="bilinear"):
    cam = GR.Camera(w._cam, dtype)
    xd = x.detach().cpu().to(dtype) if isinstance(x, torch.Tensor) else None
    if xd is not None and xd.dim() == 3:
        xd = xd[:, None]
    wtd = [t.cpu().to(dtype) for t in wt] if method == "homography" else wt.cpu().to(dtype).reshape(xd.shape[0], -1, cam.H, cam.W)
    wHd = wH.cpu().to(dtype) if wH is not None else None

    def loss(g, a):
        if method == "homography":
            H, R, Hi = GR.build_homography(cam, g, a)
            return (H * wtd[0]).sum() + (R * wtd[1]).sum() + (Hi * wtd[2]).sum()
        Hm, y = (GR.warp(cam, xd, g, a, mode) if method == "warp" else GR.inverse_warp(cam, xd, g, a))
        return (y * wtd).sum() + ((Hm * wHd).sum() if wHd is not None else 0.0)
    return GR.gravity_grads(loss, I_g, I_a, dtype)


def _rel(got, ref):
    return np.linalg.norm(got - ref, axis=1) / np.maximum(np.linalg.norm(ref, axis=1), 1e-30)


def _inputs(method, cam_name, kind, C_=3, B=3, seed=5):
    w = _warper(cam_name)
    H, W = int(w.H), int(w.W)
    I_g, I_a = C.random_gravity(B, seed=seed, roll_deg=30, pitch_deg=30)
    if method == "homography":
        wt = [torch.from_numpy(_noise((B, 3, 3), seed + k)).to(DEV) for k in range(3)]
        return w, None, I_g, I_a, wt
    C_ = 3 if method == "inverse" else C_
    x = torch.from_numpy((_smooth if kind == "smooth" else _noise)((B, C_, H, W), seed)).to(DEV)
    wt = torch.from_numpy(_smooth((B, C_, H, W), seed + 1) if kind == "smooth" else _noise((B, C_, H, W), seed + 1)).to(DEV)
    return w, x, I_g, I_a, wt


@pytest.mark.parametrize("cam_name", ["tiny", "S1", "S2"])
@pytest.mark.parametrize("method", ["warp", "inverse", "homography"])
@pytest.mark.parametrize("kind", ["smooth", "noise"])
def test_gravity_grad_accuracy(cam_name, method, kind):
    w, x, I_g, I_a, wt = _inputs(method, cam_name, kind)
    wH = None if method == "homography" else torch.from_numpy(_noise((3, 3, 3), 11)).to(DEV)
    got = _ours(w, method, x, I_g, I_a, wt, wH)
    truth = _reference(w, method, x, I_g, I_a, wt, wH, torch.float64)
    ref32 = _reference(w, method, x, I_g, I_a, wt, wH, torch.float32)
    ref = truth if kind == "smooth" else ref32
    for name, k in (("I_g", 0), ("I_a", 1)):
        err = _rel(got[k], ref[k])
        print(f"{cam_name} {method} {kind} {name}: CUDA error {err.max():.2e}, fp32 restatement vs fp64 {_rel(ref32[k], truth[k]).max():.2e}")
        assert err.max() <= TOL, (name, err, got[k], ref[k])


@pytest.mark.parametrize("layout", ["C1", "C7", "depth3d", "channels_last", "strided", "inverse"])
def test_gravity_grad_layouts_and_front_ends(layout):
    method = "inverse" if layout == "inverse" else "warp"
    C_ = {"C1": 1, "C7": 7, "depth3d": 1}.get(layout, 3)
    w, x, I_g, I_a, wt = _inputs(method, "S1", "smooth", C_=C_)
    if layout == "depth3d":
        x, wt = x[:, 0], wt[:, 0]
    elif layout == "channels_last":
        x = x.contiguous(memory_format=torch.channels_last)
    elif layout == "strided":
        big = torch.zeros(x.shape[0], 5, x.shape[2] + 3, x.shape[3] + 7, device=DEV)
        big[:, 1:4, 2:-1, 3:-4] = x
        x = big[:, 1:4, 2:-1, 3:-4]
        assert not x.is_contiguous()
        wt = wt.transpose(2, 3).contiguous().transpose(2, 3)         # a strided upstream gradient
    got = _ours(w, method, x, I_g, I_a, wt, None)
    ref = _reference(w, method, x, I_g, I_a, wt, None, torch.float64)
    for k in (0, 1):
        assert _rel(got[k], ref[k]).max() <= TOL, (layout, got[k], ref[k])


def test_nearest_and_cg_h_c_upstream():
    w, x, I_g, I_a, wt = _inputs("warp", "S1", "smooth")
    gz = _ours(w, "warp", x, I_g, I_a, wt, None, mode="nearest")
    rz = _reference(w, "warp", x, I_g, I_a, wt, None, torch.float64, mode="nearest")
    for k in (0, 1):
        assert np.array_equal(gz[k], np.zeros_like(gz[k])) and np.array_equal(rz[k], np.zeros_like(rz[k]))
    wH = torch.from_numpy(_noise((3, 3, 3), 12)).to(DEV)
    got = _ours(w, "warp", x, I_g, I_a, wt, wH, mode="nearest")
    ref = _reference(w, "warp", x, I_g, I_a, wt, wH, torch.float64, mode="nearest")
    for k in (0, 1):
        assert _rel(got[k], ref[k]).max() <= TOL


@pytest.mark.parametrize("method", ["warp", "inverse"])
def test_gravity_grad_is_bit_reproducible(method):
    w, x, I_g, I_a, wt = _inputs(method, "S2", "noise", B=5, seed=9)
    runs = [_ours(w, method, x, I_g, I_a, wt, None) for _ in range(2)]
    for k in (0, 1):
        assert np.array_equal(runs[0][k], runs[1][k])
    # frame 2 alone and at position 4 of a batch of 5
    alone = _ours(w, method, x[2:3].contiguous(), I_g[2:3], I_a[2:3], wt[2:3].contiguous(), None)
    perm = [0, 1, 3, 4, 2]
    moved = _ours(w, method, x[perm].contiguous(), I_g[perm], I_a[perm], wt[perm].contiguous(), None)
    for k in (0, 1):
        assert np.array_equal(alone[k][0], runs[0][k][2]) and np.array_equal(moved[k][4], runs[0][k][2])
    # a NaN-gravity frame leaves its neighbours' bits unchanged
    g_nan = I_g.copy()
    g_nan[1] = np.nan
    nan_run = _ours(w, method, x, g_nan, I_a, wt, None)
    for k in (0, 1):
        assert np.array_equal(np.delete(nan_run[k], 1, 0), np.delete(runs[0][k], 1, 0))


@pytest.mark.parametrize("method", ["warp", "inverse"])
def test_image_grad_unchanged_by_gravity_grad(method):
    w, x, I_g, I_a, wt = _inputs(method, "S1", "noise")
    w.deterministic_backward = True
    grads = []
    for grav in (False, True):
        xr = x.clone().requires_grad_(True)
        g = torch.from_numpy(I_g).to(DEV).requires_grad_(grav)
        a = torch.from_numpy(I_a).to(DEV).requires_grad_(grav)
        fn = w.warp_with_gravity_center_aligned if method == "warp" else w.inverse_warp_normal_image_with_gravity_center_aligned
        _, y = fn(xr, g, a)
        (y * wt).sum().backward()
        grads.append(xr.grad.cpu().numpy())
        assert (g.grad is not None) == grav
    assert C.count_bit_mismatches(grads[0], grads[1]) == 0


def _forward_only_calls(w, x3, x4, d, g, a):
    Hm = w._build_homography(g.detach(), a.detach())[0].requires_grad_(True)
    tracks = torch.zeros((x3.shape[0], 4, 4), dtype=torch.float64, device=DEV)
    p = w.prepare(g, a)
    return {
        "warp_rgbd": lambda: w.warp_rgbd(x3, d, g, a)[1],
        "warp_rgbd_H": lambda: w.warp_rgbd(x3, d, g, a)[0],
        "warp_rgbd_params": lambda: w.warp_rgbd(x3, d, params=p)[1],
        "prepare_H": lambda: p.H,
        "unwarp_normals": lambda: w.unwarp_normals(x3, g, a)[1],
        "unwarp_normals_raw": lambda: w.unwarp_normals(x3, g, a, normalize=False)[1],
        "unwarp_normals_valid": lambda: w.unwarp_normals(x3, g, a, with_valid=True)[1],
        "unwarp_normals_params": lambda: w.unwarp_normals(x3, params=p)[1],
        "warp_rgb_sparse_depth": lambda: w.warp_rgb_sparse_depth(x3, tracks, None, (1.0, 1.0), (0.0, 0.0), g, a)[1],
        "warp_rgbd_packed": lambda: w.warp_rgbd_packed(x4.contiguous(memory_format=torch.channels_last), g, a)[1],
        "image_sampler_forward_inverse": lambda: w.image_sampler_forward_inverse(g, a)[1],
        "warp_normal_image": lambda: w.warp_normal_image_with_gravity_center_aligned(x3, g, a)[1],
        "warp_with_homography": lambda: w.warp_with_homography(x3, Hm)[1],
        "bicubic": lambda: w.warp_with_gravity_center_aligned(x3, g, a, interp_mode="bicubic")[1],
        "bicubic_H": lambda: w.warp_with_gravity_center_aligned(x3, g, a, interp_mode="bicubic")[0],
    }


@pytest.mark.parametrize("name", ["warp_rgbd", "warp_rgbd_H", "warp_rgbd_params", "prepare_H", "unwarp_normals",
                                  "unwarp_normals_raw", "unwarp_normals_valid", "unwarp_normals_params", "warp_rgb_sparse_depth",
                                  "warp_rgbd_packed", "image_sampler_forward_inverse", "warp_normal_image",
                                  "warp_with_homography", "bicubic", "bicubic_H"])
def test_forward_only_entry_points_raise(name):
    w = _warper("S1")
    H, W = int(w.H), int(w.W)
    I_g, I_a = C.random_gravity(2, seed=3)
    g = torch.from_numpy(I_g).to(DEV).requires_grad_(True)
    a = torch.from_numpy(I_a).to(DEV).requires_grad_(True)
    x3 = torch.from_numpy(_noise((2, 3, H, W), 1)).to(DEV)
    x4 = torch.from_numpy(_noise((2, 4, H, W), 2)).to(DEV)
    d = torch.from_numpy(_noise((2, 1, H, W), 3)).to(DEV)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        out = _forward_only_calls(w, x3, x4, d, g, a)[name]()
        assert out.requires_grad
        with pytest.raises(NotImplementedError):
            out.sum().backward()
