"""The default (atomic) image backward of the two reference-shaped warps, vidc_warp_backward, against exact sums of its terms.

The kernel scatters each term w_tap * g into grad_in with atomicAdd, so an element is an fp32 sum of its terms in an order
that changes from run to run.  tests/exact_reference.py forms the same terms from the CPU oracle's grids and gives, per
element, their count k, exact sum E, magnitude sum A and special values; exact_reference.check_atomic_sum then holds every
element to what a sum in any order can be: +0 with no term, the order-free bits with one or two terms, the IEEE result with
NaN or infinite terms, and |S - E| <= gamma_{k-1} A (+ slack for fp64 rounding and flushed subnormals) otherwise.  Run with
-s to see the largest |S - E| / (gamma_{k-1} A) of each case (elements of three or more terms) and what the atomics did
with an element's single subnormal term (on a B200 the fp32 atomicAdd flushes it to zero)."""
import os
import time

import numpy as np
import pytest
import torch

from tests import common as C
from tests import exact_reference as X
from tests.test_gpu_backward_ordered import _call, _grad, _mk, _t

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _report(S, st, what, ratio):
    """Print the bound ratio and, for elements whose only term is subnormal, whether the atomic add kept or flushed it."""
    sub = (st["k"] == 1) & ((st["flags"] & X.F_SUBNORMAL) != 0)
    kept = int((C.bits(S)[sub] == C.bits(st["pair"])[sub]).sum())
    flushed = int(((C.bits(S)[sub] & np.uint32(0x7FFFFFFF)) == 0).sum())
    print(f"[atomic-backward] {what}: max |S-E|/(gamma A) = {ratio:.4g}; single subnormal terms kept {kept}, flushed {flushed}")


def _check(w, o, gout_np, I_g, I_a, dev, inverse, mode, in_hw=None, what="", gout=None):
    """vidc_warp_backward on gout (default: gout_np as a contiguous device tensor) against the exact statistics of gout_np."""
    g = _t(gout_np, dev) if gout is None else gout
    S = _call(w, g, _t(I_g, dev), _t(I_a, dev), inverse, mode, in_hw, entry="vidc_warp_backward").cpu().numpy()
    with np.errstate(all="ignore"):
        st = X.scatter_stats(o, gout_np, I_g, I_a, in_hw=in_hw, inverse=inverse, interp_mode=mode)
    what = f"{what} inverse={inverse} mode={mode} in_hw={in_hw}"
    ratio = X.check_atomic_sum(S, st, what)
    _report(S, st, what, ratio)
    return ratio


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_tiny_frames(cuda_device, mode):
    """Edge-case, random and golden frames at 64x48; C = 1, 3, 4 forward, 3 inverse."""
    w, o = _mk("tiny")
    H, W = int(w.H), int(w.W)
    g_e, a_e = C.edge_case_gravity()
    g_r, a_r = C.random_gravity(6, seed=4242)
    gb = np.load(os.path.join(GOLD, "golden_tiny_backward.npz"))
    I_g = np.concatenate([g_e, g_r, gb["I_g"]]); I_a = np.concatenate([a_e, a_r, gb["I_a"]])
    B = I_g.shape[0]
    for inverse in (False, True):
        for Cc in ((1, 3, 4) if not inverse else (3,)):
            _check(w, o, _grad(B, Cc, H, W, 10 + Cc), I_g, I_a, cuda_device, inverse, mode, what=f"tiny C={Cc}")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_special_values_and_degenerate_gravity(cuda_device, mode):
    """Signed zeros, subnormals, 1e35, inf and NaN in the upstream gradient; zero / NaN / inf / huge gravity; frames whose
    projective denominator is exactly zero at one pixel."""
    w, o = _mk("tiny")
    H, W = int(w.H), int(w.W)
    rgb, depth, normals = C.special_value_images(4, H, W, seed=3)
    I_g, I_a = C.special_value_gravity(4)
    for inverse, gout in ((False, rgb), (False, depth[:, None]), (True, normals), (False, normals)):
        _check(w, o, gout, I_g, I_a, cuda_device, inverse, mode, what="special values")
    g_d, a_d = C.degenerate_gravity()
    gout = _grad(g_d.shape[0], 3, H, W, 7)
    for inverse in (False, True):
        _check(w, o, gout, g_d, a_d, cuda_device, inverse, mode, what="degenerate gravity")
    w1, o1 = _mk("S1")
    g_i, a_i = C.isolated_nonfinite_gravity()
    gout = _grad(g_i.shape[0], 3, int(w1.H), int(w1.W), 8)
    for inverse in (False, True):
        _check(w1, o1, gout, g_i, a_i, cuda_device, inverse, mode, what="isolated non-finite")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_full_resolution(cuda_device, mode):
    """S1 (320x240), S2 (640x480), S3 at rolls 0, +-45, +-90 deg, and a 640x489 canvas."""
    for cam, B, grav in (("S1", 4, C.random_gravity(4, seed=31)), ("S2", 2, C.random_gravity(2, seed=32, roll_deg=40, pitch_deg=35))):
        w, o = _mk(cam)
        for inverse in (False, True):
            _check(w, o, _grad(B, 3, int(w.H), int(w.W), 5), *grav, cuda_device, inverse, mode, what=cam)
    w, o = _mk("S3")
    rolls = np.deg2rad(np.array([0, 45, -45, 90, -90], np.float32))
    I_g = C.gravity_from_angles(rolls, np.zeros(5, np.float32))
    I_a = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (5, 1))
    for inverse in (False, True):
        _check(w, o, _grad(5, 3, int(w.H), int(w.W), 6), I_g, I_a, cuda_device, inverse, mode, what="S3 rolls")
    w, o = _mk((404.0, 404.0, 319.87654, 244.4))
    assert (int(w.W), int(w.H)) == (640, 489)
    I_g, I_a = C.random_gravity(2, seed=33, roll_deg=60, pitch_deg=20)
    for inverse in (False, True):
        _check(w, o, _grad(2, 3, 489, 640, 9), I_g, I_a, cuda_device, inverse, mode, what="640x489")


@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_input_size_differs_from_canvas(cuda_device, mode):
    """Inputs larger and smaller than the canvas; at 7x9 thousands of terms land on each element."""
    w, o = _mk("S1")
    I_g, I_a = C.random_gravity(3, seed=41, roll_deg=50, pitch_deg=30)
    for in_hw in ((483, 635), (121, 107), (7, 9)):
        for Cc in (1, 4):
            _check(w, o, _grad(3, Cc, 240, 320, 11), I_g, I_a, cuda_device, False, mode, in_hw=in_hw, what=f"in size C={Cc}")
    big = np.random.RandomState(12).randn(3, 1, 240, 320).astype(np.float32) * np.float32(1e35)      # some orders overflow
    _check(w, o, big, I_g, I_a, cuda_device, False, mode, in_hw=(7, 9), what="1e35 upsampled")


def test_strided_grad_out(cuda_device):
    """Channels-last, channel-sliced and stride-0 (expand) upstream gradients."""
    w, o = _mk("S1")
    I_g, I_a = C.random_gravity(2, seed=43, roll_deg=60, pitch_deg=30)
    big = _t(_grad(2, 6, 240, 320, 12), cuda_device)
    row = _t(_grad(2, 3, 1, 320, 13), cuda_device)
    for inverse in (False, True):
        for mode in (("bilinear", "nearest") if not inverse else ("bilinear",)):
            sl = big[:, 1:4]
            for name, gout in (("channels-last", sl.contiguous(memory_format=torch.channels_last)), ("channel-sliced", sl),
                               ("expand", row.expand(2, 3, 240, 320))):
                _check(w, o, gout.cpu().numpy(), I_g, I_a, cuda_device, inverse, mode, what=name, gout=gout)


def test_random_cameras(cuda_device):
    """A bounded random search: canvases of 40..400 px, any roll, pitch up to 80 deg, inputs of other sizes, 1..4 channels."""
    rs = np.random.RandomState(2027)
    t_end = time.time() + 20.0
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
        _check(w, o, _grad(B, Cc, int(w.H), int(w.W), n), I_g, I_a, cuda_device, inverse, mode, in_hw=in_hw,
               what=f"random case {n} cam={cam}")
        n += 1


def _autograd_grad(w, dev, x_np, I_g, I_a, method, mode, wt_np):
    """x.grad through a reference-shaped method with the default (atomic) backward; wt_np None: y.sum().backward()."""
    x = _t(x_np, dev).requires_grad_(True)
    g, a = _t(I_g, dev), _t(I_a, dev)
    if method == "inverse":
        _, y = w.inverse_warp_normal_image_with_gravity_center_aligned(x, g, a)
    else:
        _, y = w.warp_with_gravity_center_aligned(x, g, a, interp_mode=mode)
    (y.sum() if wt_np is None else (y * _t(wt_np, dev)).sum()).backward()
    return x.grad.cpu().numpy()


def test_autograd_through_the_reference_shaped_methods(cuda_device):
    """Both methods, bilinear and nearest, 3-D depth, a 7-channel map (plane groups of at most four), y.sum().backward()
    (an all-zero-stride gradient), and a batch holding a NaN-gravity frame and a NaN-gradient frame next to finite ones."""
    assert not torch.are_deterministic_algorithms_enabled()
    w, o = _mk("S1")
    assert w.deterministic_backward is None
    H, W = int(w.H), int(w.W)
    I_g, I_a = C.random_gravity(3, seed=21, roll_deg=50, pitch_deg=30)
    rs = np.random.RandomState(4)
    x3, x7 = rs.rand(3, 3, H, W).astype(np.float32), rs.rand(3, 7, H, W).astype(np.float32)
    wt3, wt7 = rs.randn(3, 3, H, W).astype(np.float32), rs.randn(3, 7, H, W).astype(np.float32)
    for mode in ("bilinear", "nearest"):
        for name, x, wt in (("C=3", x3, wt3), ("C=7", x7, wt7), ("3-D depth", x3[:, 0], wt3[:, 0]), ("sum", x3, None)):
            got = _autograd_grad(w, cuda_device, x, I_g, I_a, "forward", mode, wt)
            gout = np.ones(x.shape, np.float32) if wt is None else wt
            st = X.scatter_stats(o, gout, I_g, I_a, interp_mode=mode)
            what = f"autograd forward {name} {mode}"
            _report(got, st, what, X.check_atomic_sum(got, st, what))
    for name, wt in (("inverse", wt3), ("inverse sum", None)):
        got = _autograd_grad(w, cuda_device, x3, I_g, I_a, "inverse", "bilinear", wt)
        st = X.scatter_stats(o, np.ones(x3.shape, np.float32) if wt is None else wt, I_g, I_a, inverse=True)
        _report(got, st, name, X.check_atomic_sum(got, st, name))
    I_gn = I_g.copy(); I_gn[1] = np.nan
    wtn = wt3.copy(); wtn[2, :, 50:60] = np.nan
    for method in ("forward", "inverse"):
        got = _autograd_grad(w, cuda_device, x3, I_gn, I_a, method, "bilinear", wtn)
        with np.errstate(all="ignore"):
            st = X.scatter_stats(o, wtn, I_gn, I_a, inverse=method == "inverse")
        what = f"autograd {method} with NaN frames"
        _report(got, st, what, X.check_atomic_sum(got, st, what))
        assert (C.bits(got[1]) == 0).all() and np.isfinite(got[0]).all() and np.isnan(got[2]).any()
