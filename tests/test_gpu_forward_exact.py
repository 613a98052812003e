"""Bit-exact references for the two forward warps that have no serial restatement in the oracle:

- the rotated forward warp, warp_normal_image_with_gravity_center_aligned: the oracle's forward warp of the normals followed
  by z = R y as the kernel computes it (k-ascending FMA chain from +0; tests/exact_reference.py: rotate);
- the explicit-homography warp, warp_with_homography: frame_params_from_h_kernel's fp64 parameter block restated in numpy,
  the fp32 coordinate chain of the forward kernels (exact_reference.homography_grid), then the oracle's bilinear sampler.

The fp64 checks of intent stay in test_gpu_parity.py."""
import os
import sys

import numpy as np
import pytest
import torch

if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests import common as C
from tests import exact_reference as X

pytestmark = pytest.mark.gpu
CANVASES = {"S1": C.CAMERAS["S1"], "S2": C.CAMERAS["S2"], "201x141": (120.0, 118.0, 100.3, 70.2)}


def _mk(intr):
    from oracle import oracle as O
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    return Warping2DOFAlignment(*intr), O.Oracle(*intr)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _kernels_child():
    """Run in a fresh process (profiler sessions are kept out of the test process): the kernels each warp launches."""
    import json
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    dev = torch.device("cuda", 0)
    w, o = _mk(C.CAMERAS["S2"])
    I_g, I_a = C.random_gravity(2, seed=3)
    g, a = _t(I_g, dev), _t(I_a, dev)
    x = _t(C.random_images(2, o.H, o.W, 1)[2], dev)
    p = w.prepare(g, a)
    calls = {"rotated": lambda: w.warp_normal_image_with_gravity_center_aligned(x, g, a),
             "homography": lambda: w.warp_with_homography(x, p.H[:1])}
    seen = {}
    for name, fn in [("warm-up", calls["rotated"])] + list(calls.items()):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        seen[name] = [e.name.split("(")[0].removeprefix("void ").removeprefix("vidc_k::").strip() for e in prof.events()
                      if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memset", "Memcpy")) and "at::" not in e.name]
    print(json.dumps(seen), flush=True)


def test_kernels_reached(cuda_device):
    """The rotated forward warp runs the generic forward kernel with the rotation; the explicit-homography warp builds its
    parameters with frame_params_from_h_kernel, then runs the generic forward kernel without it."""
    import json
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--kernels"], cwd=root, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    seen = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert seen["rotated"] == ["frame_params_kernel", "warp_forward_kernel<3, false, true>"], seen
    assert seen["homography"] == ["frame_params_from_h_kernel", "warp_forward_kernel<3, false, false>"], seen
    print(f"[forward exact] kernels: {seen}")


def _variants(x_np, dev):
    """The same images as a contiguous tensor, channels-last, and a column-strided view of a wider buffer."""
    x = _t(x_np, dev)
    wide = torch.zeros(*x.shape[:3], 2 * x.shape[3], device=dev)
    wide[..., 1::2] = x
    return [("contiguous", x), ("channels-last", x.contiguous(memory_format=torch.channels_last)), ("strided", wide[..., 1::2])]


def _rotated_expect(o, x_np, I_g, I_a, mode):
    with np.errstate(all="ignore"):
        H, y = o.warp_with_gravity_center_aligned(x_np, I_g, I_a, interp_mode=mode)
        _, R, _ = o.build_homography(I_g, I_a)
        return H, X.rotate(y, R)


def _check_rotated(w, o, x_np, I_g, I_a, dev, mode, what, variants=True):
    wantH, want = _rotated_expect(o, x_np, I_g, I_a, mode)
    for name, x in (_variants(x_np, dev) if variants else [("contiguous", _t(x_np, dev))]):
        H, z = w.warp_normal_image_with_gravity_center_aligned(x, _t(I_g, dev), _t(I_a, dev), interp_mode=mode)
        assert z.is_contiguous(memory_format=torch.channels_last if name == "channels-last" else torch.contiguous_format), (what, name)
        assert C.count_bit_mismatches(H.cpu().numpy(), wantH) == 0, (what, name, mode, "Cg_H_C")
        n = C.count_bit_mismatches(z.cpu().numpy(), want)
        assert n == 0, f"{what} {name} {mode}: {n} elements differ from R y"


@pytest.mark.parametrize("mode", ["bilinear", "nearest", "bicubic"])
def test_rotated_forward_warp_bit_exact(cuda_device, mode):
    """S1, S2 and a 201x141 canvas; edge-case and extreme-roll gravity; inputs of the canvas size, larger and smaller;
    contiguous, channels-last and column-strided inputs (the output's memory format follows the input)."""
    for cname, intr in CANVASES.items():
        w, o = _mk(intr)
        g_e, a_e = C.edge_case_gravity()
        g_x, a_x = C.extreme_roll_gravity(7, 3)
        I_g, I_a = np.concatenate([g_e[:6], g_x]), np.concatenate([a_e[:6], a_x])
        B = I_g.shape[0]
        for hw in ((o.H, o.W), (o.H + 37, o.W + 91), (o.H // 2 + 3, o.W // 3 + 1)):
            x = C.random_images(B, hw[0], hw[1], 11)[2]
            _check_rotated(w, o, x, I_g, I_a, cuda_device, mode, f"{cname} in={hw}", variants=hw == (o.H, o.W) or cname == "201x141")


@pytest.mark.parametrize("mode", ["bilinear", "nearest", "bicubic"])
def test_rotated_forward_warp_special_values(cuda_device, mode):
    """Special-value images, degenerate gravity, a frame with R = I whose -0 inputs must come out +0, and B = 0."""
    w, o = _mk(C.CAMERAS["S1"])
    x = C.special_value_images(4, o.H, o.W, 21)[2]
    I_g, I_a = C.special_value_gravity(4)
    _, R, _ = o.build_homography(I_g, I_a)
    assert np.array_equal(R[0], np.eye(3, dtype=np.float32))
    x[0, :, :20] = -0.0
    _check_rotated(w, o, x, I_g, I_a, cuda_device, mode, "special values")
    _, z = w.warp_normal_image_with_gravity_center_aligned(_t(x, cuda_device), _t(I_g, cuda_device), _t(I_a, cuda_device), interp_mode=mode)
    z0 = z[0].cpu().numpy()
    assert (z0 == 0).any() and not (np.signbit(z0) & (z0 == 0)).any()
    g_d, a_d = C.degenerate_gravity()
    xd = C.random_images(g_d.shape[0], o.H, o.W, 12)[2]
    _check_rotated(w, o, xd, g_d, a_d, cuda_device, mode, "degenerate gravity", variants=False)
    g0 = torch.zeros(0, 3, device=cuda_device)
    H, z = w.warp_normal_image_with_gravity_center_aligned(torch.zeros(0, 3, o.H, o.W, device=cuda_device), g0, g0, interp_mode=mode)
    assert H.shape == (0, 3, 3) and z.shape == (0, 3, o.H, o.W)


def _homographies(o):
    """Moderate, steep-pitch and +-90 deg roll frames."""
    g_r, a_r = C.random_gravity(2, seed=19, roll_deg=25, pitch_deg=20)
    g_p, a_p = C.random_gravity(2, seed=20, roll_deg=10, pitch_deg=75)
    g_x, a_x = C.extreme_roll_gravity(7, 3)
    Hm, _, _ = o.build_homography(np.concatenate([g_r, g_p, g_x[[5, 6]]]), np.concatenate([a_r, a_p, a_x[[5, 6]]]))
    return Hm


@pytest.mark.parametrize("cname", ["S1", "201x141"])
def test_explicit_homography_warp_bit_exact(cuda_device, cname):
    """C = 1..4; per-frame (B,3,3) homographies as a device tensor and as numpy; inputs of the canvas size, larger and
    smaller; contiguous, channels-last and column-strided inputs."""
    w, o = _mk(CANVASES[cname])
    Hm = _homographies(o)
    B = Hm.shape[0]
    for Cc in (1, 2, 3, 4):
        for hw in ((o.H, o.W), (o.H + 29, o.W + 53), (o.H // 2 + 5, o.W // 2 - 3)):
            x_np = np.random.RandomState(Cc).rand(B, Cc, *hw).astype(np.float32)
            want = X.warp_with_homography(o, w._cam, x_np, Hm)
            for name, x in _variants(x_np, cuda_device):
                for hname, h in (("tensor", torch.from_numpy(Hm).to(cuda_device)), ("numpy", Hm)):
                    _, y = w.warp_with_homography(x, h)
                    n = C.count_bit_mismatches(y.cpu().numpy(), want)
                    assert n == 0, f"{cname} C={Cc} in={hw} {name} {hname}: {n} elements differ"


def test_explicit_homography_broadcast(cuda_device):
    """One (1,3,3) homography for the whole batch, as a device tensor and as numpy."""
    w, o = _mk(C.CAMERAS["S2"])
    Hm = _homographies(o)
    for k in range(Hm.shape[0]):
        x_np = np.random.RandomState(k).rand(3, 3, o.H, o.W).astype(np.float32)
        want = X.warp_with_homography(o, w._cam, x_np, np.repeat(Hm[k:k + 1], 3, 0))
        for h in (torch.from_numpy(Hm[k:k + 1]).to(cuda_device), Hm[k:k + 1]):
            _, y = w.warp_with_homography(_t(x_np, cuda_device), h)
            assert C.count_bit_mismatches(y.cpu().numpy(), want) == 0, k


if __name__ == "__main__" and sys.argv[1:2] == ["--kernels"]:
    _kernels_child()
