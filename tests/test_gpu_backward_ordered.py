"""The fixed-order backward of the two warps (vidc_warp_backward_ordered) against its serial restatement
(tests/backward_oracle.py over the CPU oracle's grids): zero differing bits, for bilinear and nearest, forward and inverse warp, over the edge cases the
forward kernels are pinned on; reproducibility; complete writes; selection through torch.use_deterministic_algorithms and
Warping2DOFAlignment.deterministic_backward; argument errors."""
import ctypes
import os
import time

import numpy as np
import pytest
import torch

from tests import backward_oracle as BO
from tests import common as C

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MODES = {"bilinear": 0, "nearest": 1}


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _mk(cam, dev=None):
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    from oracle import oracle as O
    fx, fy, cx, cy = C.CAMERAS[cam] if isinstance(cam, str) else cam
    return Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy), O.Oracle(fx, fy, cx, cy)


def _call(w, gout, g, a, inverse, mode, in_hw=None, out=None, entry="vidc_warp_backward_ordered"):
    """One call of the C entry point on the current stream; gout (B,C,H,W) any strides, g / a (B,3) device tensors."""
    from vi_depth_completion_b200._cabi import check, lib
    from vi_depth_completion_b200.warping_2dof_alignment import _image, _stream_ptr
    dev = gout.device
    B, Cc = gout.shape[:2]
    Hin, Win = (int(w.H), int(w.W)) if in_hw is None else in_hw
    if out is None:
        out = torch.empty((B, Cc, Hin, Win), dtype=torch.float32, device=dev)
    gi = _image(gout)
    ws = w._params_ws(max(B, 1), dev)
    check(getattr(lib(), entry)(ctypes.byref(w._cam), ctypes.byref(gi), g.data_ptr(), a.data_ptr(), g.shape[0], 1 if inverse else 0,
                                MODES[mode], ws.data_ptr(), out.data_ptr(), Hin, Win, _stream_ptr(dev)))
    return out


def _assert_bits(w, o, gout_np, I_g, I_a, dev, inverse, mode, in_hw=None, what=""):
    got = _call(w, _t(gout_np, dev), _t(I_g, dev), _t(I_a, dev), inverse, mode, in_hw).cpu().numpy()
    want = BO.warp_backward(o, gout_np, I_g, I_a, in_hw=in_hw, inverse=inverse, interp_mode=mode)
    assert got.shape == want.shape
    n = C.count_bit_mismatches(got, want)
    assert n == 0, f"{what} inverse={inverse} mode={mode} in_hw={in_hw}: {n} elements differ from the oracle"
    return got, want


def _grad(B, Cc, H, W, seed):
    return np.random.RandomState(seed).randn(B, Cc, H, W).astype(np.float32)


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_tiny_frames_bit_exact(cuda_device, mode):
    w, o = _mk("tiny")
    H, W = int(w.H), int(w.W)
    g_e, a_e = C.edge_case_gravity()
    g_r, a_r = C.random_gravity(6, seed=4242)
    gb = np.load(os.path.join(GOLD, "golden_tiny_backward.npz"))
    I_g = np.concatenate([g_e, g_r, gb["I_g"]]); I_a = np.concatenate([a_e, a_r, gb["I_a"]])
    B = I_g.shape[0]
    for inverse in (False, True):
        for Cc in ((1, 3, 4) if not inverse else (3,)):
            _assert_bits(w, o, _grad(B, Cc, H, W, 10 + Cc), I_g, I_a, cuda_device, inverse, mode, what=f"tiny C={Cc}")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_special_values_and_degenerate_gravity(cuda_device, mode):
    """Signed zeros, denormals, inf and NaN in the upstream gradient; zero / NaN / inf / huge gravity (non-finite coordinates
    contribute nothing); frames whose projective denominator is exactly zero at one pixel."""
    w, o = _mk("tiny")
    H, W = int(w.H), int(w.W)
    rgb, depth, normals = C.special_value_images(4, H, W, seed=3)
    I_g, I_a = C.special_value_gravity(4)
    for inverse, gout in ((False, rgb), (False, depth[:, None]), (True, normals), (False, normals)):
        _assert_bits(w, o, gout, I_g, I_a, cuda_device, inverse, mode, what="special values")
    g_d, a_d = C.degenerate_gravity()
    gout = _grad(g_d.shape[0], 3, H, W, 7)
    for inverse in (False, True):
        _assert_bits(w, o, gout, g_d, a_d, cuda_device, inverse, mode, what="degenerate gravity")
    w1, o1 = _mk("S1")
    g_i, a_i = C.isolated_nonfinite_gravity()
    gout = _grad(g_i.shape[0], 3, int(w1.H), int(w1.W), 8)
    for inverse in (False, True):
        _assert_bits(w1, o1, gout, g_i, a_i, cuda_device, inverse, mode, what="isolated non-finite")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_full_resolution_bit_exact(cuda_device, mode):
    """S1 (320x240, 4 frames), S2 (640x480, 2 frames), S3 at rolls 0, +-45, +-90 deg, and a 640x489 canvas."""
    for cam, B, grav in (("S1", 4, C.random_gravity(4, seed=31)), ("S2", 2, C.random_gravity(2, seed=32, roll_deg=40, pitch_deg=35))):
        w, o = _mk(cam)
        for inverse in (False, True):
            _assert_bits(w, o, _grad(B, 3, int(w.H), int(w.W), 5), *grav, cuda_device, inverse, mode, what=cam)
    w, o = _mk("S3")
    rolls = np.deg2rad(np.array([0, 45, -45, 90, -90], np.float32))
    I_g = C.gravity_from_angles(rolls, np.zeros(5, np.float32))
    I_a = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (5, 1))
    for inverse in (False, True):
        _assert_bits(w, o, _grad(5, 3, int(w.H), int(w.W), 6), I_g, I_a, cuda_device, inverse, mode, what="S3 rolls")
    w, o = _mk((404.0, 404.0, 319.87654, 244.4))
    assert (int(w.W), int(w.H)) == (640, 489)
    I_g, I_a = C.random_gravity(2, seed=33, roll_deg=60, pitch_deg=20)
    for inverse in (False, True):
        _assert_bits(w, o, _grad(2, 3, 489, 640, 9), I_g, I_a, cuda_device, inverse, mode, what="640x489")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_input_size_differs_from_canvas(cuda_device, mode):
    """Forward warp of inputs larger and smaller than the canvas; a 9x7 input makes every tap origin receive far more output
    pixels than a list holds (the chunk-rescan path)."""
    w, o = _mk("S1")
    I_g, I_a = C.random_gravity(3, seed=41, roll_deg=50, pitch_deg=30)
    for in_hw in ((2 * 240 + 3, 2 * 320 - 5), (121, 107), (7, 9), (240, 320)):
        for Cc in (1, 4):
            _assert_bits(w, o, _grad(3, Cc, 240, 320, 11), I_g, I_a, cuda_device, False, mode, in_hw=in_hw, what="in size")


def test_strided_grad_out(cuda_device):
    """Channels-last and channel-sliced upstream gradients give the bits of the contiguous one."""
    w, o = _mk("S1")
    I_g, I_a = C.random_gravity(2, seed=43)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    big = _t(_grad(2, 6, 240, 320, 12), cuda_device)
    for inverse in (False, True):
        for mode in (("bilinear", "nearest") if not inverse else ("bilinear",)):
            ref = _call(w, big[:, 1:4].contiguous(), g, a, inverse, mode)
            cl = big[:, 1:4].contiguous(memory_format=torch.channels_last)
            assert torch.equal(_call(w, cl, g, a, inverse, mode), ref)
            assert torch.equal(_call(w, big[:, 1:4], g, a, inverse, mode), ref)
            want = BO.warp_backward(o, big[:, 1:4].cpu().numpy(), I_g, I_a, inverse=inverse, interp_mode=mode)
            assert C.count_bit_mismatches(ref.cpu().numpy(), want) == 0


def test_random_cameras(cuda_device):
    """A bounded random search: canvases of 40..400 px, any roll, pitch up to 80 deg, inputs of other sizes, 1..4 channels."""
    rs = np.random.RandomState(2026)
    t_end = time.time() + 30.0
    n = 0
    while time.time() < t_end or n < 10:
        W, H = int(rs.randint(40, 401)), int(rs.randint(40, 401))
        f = float(rs.uniform(0.4, 1.5) * max(W, H))
        cam = (f, f * float(rs.uniform(0.9, 1.1)), (W - 0.3) / 2.0, (H - 0.3) / 2.0)
        w, o = _mk(cam)
        B = int(rs.randint(1, 4))
        roll = rs.uniform(-np.pi, np.pi, B).astype(np.float32)
        pitch = np.deg2rad(rs.uniform(-80, 80, B)).astype(np.float32)
        I_g = C.gravity_from_angles(roll, pitch)
        I_a = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (B, 1))
        inverse = bool(rs.rand() < 0.4)
        mode = "bilinear" if (inverse or rs.rand() < 0.7) else "nearest"
        Cc = 3 if inverse else int(rs.randint(1, 5))
        in_hw = None if inverse or rs.rand() < 0.5 else (int(rs.randint(8, 2 * int(w.H) + 1)), int(rs.randint(8, 2 * int(w.W) + 1)))
        _assert_bits(w, o, _grad(B, Cc, int(w.H), int(w.W), n), I_g, I_a, cuda_device, inverse, mode, in_hw=in_hw,
                     what=f"random case {n} cam={cam}")
        n += 1


def test_reproducible(cuda_device):
    """The same call twice, a frame at another batch position or alone, and a non-default stream: identical bits."""
    w, _ = _mk("S2")
    I_g, I_a = C.random_gravity(4, seed=51, roll_deg=45)
    g, a = _t(I_g, cuda_device), _t(I_a, cuda_device)
    gout = _t(_grad(4, 3, 480, 640, 13), cuda_device)
    for inverse in (False, True):
        r1 = _call(w, gout, g, a, inverse, "bilinear")
        r2 = _call(w, gout, g, a, inverse, "bilinear")
        assert torch.equal(r1, r2)
        perm = torch.tensor([2, 0, 3, 1], device=cuda_device)
        rp = _call(w, gout[perm].contiguous(), g[perm].contiguous(), a[perm].contiguous(), inverse, "bilinear")
        assert torch.equal(rp, r1[perm])
        r_one = _call(w, gout[2:3], g[2:3], a[2:3], inverse, "bilinear")
        assert torch.equal(r_one[0], r1[2])
        s = torch.cuda.Stream(cuda_device)
        s.wait_stream(torch.cuda.current_stream(cuda_device))
        with torch.cuda.stream(s):
            rs_ = _call(w, gout, g, a, inverse, "bilinear")
        torch.cuda.current_stream(cuda_device).wait_stream(s)
        assert torch.equal(rs_, r1)


def test_every_element_is_written(cuda_device):
    """Into a NaN-prefilled buffer: no NaN remains where the oracle's gradient is finite, and nothing is written outside the
    buffer (NaN guard bands on both sides stay NaN)."""
    w, o = _mk("S1")
    I_g, I_a = C.random_gravity(3, seed=61, roll_deg=70, pitch_deg=40)
    guard = 4096
    for inverse, in_hw in ((False, None), (False, (300, 411)), (False, (37, 45)), (True, None)):
        gout = _grad(3, 3, 240, 320, 14)
        Hin, Win = (240, 320) if in_hw is None else in_hw
        n = 3 * 3 * Hin * Win
        buf = torch.full((n + 2 * guard,), float("nan"), device=cuda_device)
        _call(w, _t(gout, cuda_device), _t(I_g, cuda_device), _t(I_a, cuda_device), inverse, "bilinear", in_hw,
              out=buf[guard:guard + n].view(3, 3, Hin, Win))
        want = BO.warp_backward(o, gout, I_g, I_a, in_hw=in_hw, inverse=inverse)
        host = buf.cpu().numpy()
        got = host[guard:guard + n].reshape(3, 3, Hin, Win)
        assert np.isnan(host[:guard]).all() and np.isnan(host[guard + n:]).all()
        assert not np.isnan(got[np.isfinite(want)]).any()
        assert C.count_bit_mismatches(got, want) == 0


def _autograd(w, dev, x_np, I_g, I_a, inverse, mode="bilinear", wt_np=None):
    x = _t(x_np, dev).requires_grad_(True)
    g, a = _t(I_g, dev), _t(I_a, dev)
    if inverse:
        _, y = w.inverse_warp_normal_image_with_gravity_center_aligned(x, g, a)
    else:
        _, y = w.warp_with_gravity_center_aligned(x, g, a, interp_mode=mode)
    (y * _t(wt_np, dev)).sum().backward()
    return x.grad.cpu().numpy()


def test_selected_under_deterministic_algorithms(cuda_device):
    """torch.use_deterministic_algorithms(True): autograd through both reference-shaped methods returns the oracle's bits and
    stays within 2e-5 of the gradients frozen from the reference's autograd."""
    gb = np.load(os.path.join(GOLD, "golden_tiny_backward.npz"))
    w, o = _mk(tuple(float(v) for v in gb["cam"]))
    assert w.deterministic_backward is None
    I_g, I_a = gb["I_g"], gb["I_a"]
    B, H, W = I_g.shape[0], int(w.H), int(w.W)
    rgb, depth, normals = C.random_images(B, H, W, int(gb["seed"]))
    wt = np.random.RandomState(int(gb["wt_seed"])).randn(B, 3, H, W).astype(np.float32)
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        got_rgb = _autograd(w, cuda_device, rgb, I_g, I_a, False, wt_np=wt)
        got_depth = _autograd(w, cuda_device, depth, I_g, I_a, False, wt_np=wt[:, 0])          # 3-D input
        got_inv = _autograd(w, cuda_device, normals, I_g, I_a, True, wt_np=wt)
        got_near = _autograd(w, cuda_device, rgb, I_g, I_a, False, mode="nearest", wt_np=wt)
    finally:
        torch.use_deterministic_algorithms(prev)
    assert C.count_bit_mismatches(got_rgb, BO.warp_backward(o, wt, I_g, I_a)) == 0
    assert C.count_bit_mismatches(got_depth, BO.warp_backward(o, wt[:, 0], I_g, I_a)) == 0
    assert C.count_bit_mismatches(got_inv, BO.warp_backward(o, wt, I_g, I_a, inverse=True)) == 0
    assert C.count_bit_mismatches(got_near, BO.warp_backward(o, wt, I_g, I_a, interp_mode="nearest")) == 0
    for got, name in ((got_rgb, "grad_forward_rgb"), (got_depth, "grad_forward_depth"), (got_inv, "grad_inverse_normals")):
        assert np.abs(got.astype(np.float64) - gb[name]).max() <= 2e-5, name


def test_selected_by_the_attribute_and_plane_groups(cuda_device):
    """deterministic_backward = True without the torch flag; a 7-channel map goes through plane groups and its channels 4..6
    get the 3-channel gradient bit for bit; input larger than the canvas."""
    w, o = _mk("S1")
    w.deterministic_backward = True
    assert not torch.are_deterministic_algorithms_enabled()
    I_g, I_a = C.random_gravity(3, seed=21)
    x = np.random.RandomState(4).rand(3, 7, 240, 320).astype(np.float32)
    wt = np.random.RandomState(5).randn(3, 7, 240, 320).astype(np.float32)
    g7 = _autograd(w, cuda_device, x, I_g, I_a, False, wt_np=wt)
    g3 = _autograd(w, cuda_device, np.ascontiguousarray(x[:, 4:7]), I_g, I_a, False, wt_np=np.ascontiguousarray(wt[:, 4:7]))
    assert C.count_bit_mismatches(g7[:, 4:7], g3) == 0
    assert C.count_bit_mismatches(g7, BO.warp_backward(o, wt, I_g, I_a)) == 0
    big = np.random.RandomState(6).rand(3, 2, 301, 397).astype(np.float32)
    gbig = _autograd(w, cuda_device, big, I_g, I_a, False, mode="nearest", wt_np=wt[:, :2])
    assert C.count_bit_mismatches(gbig, BO.warp_backward(o, wt[:, :2], I_g, I_a, in_hw=(301, 397), interp_mode="nearest")) == 0


def test_errors_match_the_scatter_entry_point(cuda_device):
    w, _ = _mk("tiny")
    H, W = int(w.H), int(w.W)
    g = torch.zeros(2, 3, device=cuda_device); g[:, 1] = 1
    gout = torch.zeros(2, 3, H, W, device=cuda_device)
    cases = [
        (AssertionError, dict(gout=gout, g=g[:1], a=g[:1], inverse=False)),                          # batch mismatch
        (RuntimeError, dict(gout=torch.zeros(2, 5, H, W, device=cuda_device), g=g, a=g, inverse=False)),   # > 4 planes
        (RuntimeError, dict(gout=gout, g=g, a=g, inverse=False, in_hw=(0, W))),                      # bad input size
        (RuntimeError, dict(gout=torch.zeros(2, 3, H + 1, W, device=cuda_device), g=g, a=g, inverse=False)),   # not the canvas
        (RuntimeError, dict(gout=gout[:, :2], g=g, a=g, inverse=True)),                              # inverse needs 3 channels
        (RuntimeError, dict(gout=gout, g=g, a=g, inverse=True, in_hw=(H, W + 1))),                   # inverse needs the canvas
        (RuntimeError, dict(gout=torch.zeros(1, 1, H, W, device=cuda_device).expand(65536, 1, H, W), g=g, a=g, inverse=False)),
    ]
    for exc, kw in cases:
        for entry in ("vidc_warp_backward", "vidc_warp_backward_ordered"):
            with pytest.raises(exc):
                _call(w, kw["gout"], kw["g"], kw["a"], kw["inverse"], "bilinear", kw.get("in_hw"),
                      out=torch.empty(1, device=cuda_device), entry=entry)
