"""The gravity gradient on the CPU: the torch restatement (tests/gravity_grad_reference.py) against the executed reference and
against finite differences, and the host build of the per-frame chain (csrc/frame_params_grad.cuh, the source of
vidc_frame_params_backward) against the restatement's autograd.  Runs without a GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from tests import common as C
from tests import gravity_grad_reference as GR

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


def _camera(name_or_cam):
    from vi_depth_completion_b200._cabi import VidcCamera, lib
    c = VidcCamera()
    vals = C.CAMERAS[name_or_cam] if isinstance(name_or_cam, str) else name_or_cam
    assert lib().vidc_camera_init(*[float(v) for v in vals], ctypes.byref(c)) == 0
    return c


def _ulp(a, b):
    a = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.ascontiguousarray(b, np.float32).view(np.int32).astype(np.int64)
    a = np.where(a < 0, -(a & 0x7fffffff), a)
    b = np.where(b < 0, -(b & 0x7fffffff), b)
    return np.abs(a - b)


def test_fp32_restatement_is_the_executed_reference_on_golden_tiny():
    """Parameters, both sampling grids and both warped images: the fp32 restatement must give the reference's bits.  The
    golden's grids come from image_sampler_forward_inverse, whose aspect guard (:178-187) replaces the grids of some frames;
    those frames are compared on their parameters and warped images only."""
    g = np.load(os.path.join(GOLD, "golden_tiny.npz"))
    cam = GR.Camera(_camera(g["cam"]), torch.float32)
    I_g, I_a = torch.from_numpy(g["I_g"]), torch.from_numpy(g["I_a"])
    B = I_g.shape[0]
    rgb, _, normals = C.random_images(B, cam.H, cam.W, int(g["seed"]))
    with torch.no_grad():
        p = GR.params(cam, I_g, I_a)
        _, y = GR.warp(cam, torch.from_numpy(rgb), I_g, I_a)
        _, z = GR.inverse_warp(cam, torch.from_numpy(normals), I_g, I_a)
        grids = {"grid": GR.forward_grid(cam, p).numpy(), "inv_grid": GR.inverse_grid(cam, p).numpy()}
    report = {}
    for k, gk in (("H", "Hm"), ("R", "R"), ("Hinv", "Hinv")):
        report[k] = int(_ulp(p[k].numpy(), g[gk]).max())
    unguarded = np.array([np.array_equal(g["Rt_guard"][i], g["R"][i].T) for i in range(B)])
    assert unguarded.sum() >= B // 2
    for k, v in list(grids.items()) + [("y_rgb", y.numpy()), ("z", z.numpy())]:
        assert v.shape == tuple(g[k + "_shape"]), k
        idx = g[k + "_idx"]
        keep = unguarded[idx // (v.size // B)] if k in grids else np.ones(idx.size, bool)
        report[k] = int(_ulp(v.reshape(-1)[idx][keep], g[k + "_val"][keep]).max())
    print("ulp distance of the fp32 restatement from the executed reference:", report)
    assert all(d == 0 for d in report.values()), report


def _smooth(B, C_, H, W, seed, dtype=torch.float64):
    rs = np.random.RandomState(seed)
    Y, X = np.meshgrid(np.arange(H) / H, np.arange(W) / W, indexing="ij")
    out = np.zeros((B, C_, H, W))
    for b in range(B):
        for c in range(C_):
            f = rs.uniform(1.0, 3.0, 4)
            out[b, c] = np.sin(2 * np.pi * (f[0] * X + f[1] * Y) + f[2]) + 0.5 * np.cos(2 * np.pi * f[3] * X * Y)
    return torch.tensor(out, dtype=dtype)


@pytest.mark.parametrize("inverse", [False, True])
def test_fp64_restatement_autograd_matches_finite_differences(inverse):
    """Smooth images, tilts of up to 30 degrees (no min / max ties, away from the 4:3 branch boundary)."""
    cam = GR.Camera(_camera("tiny"), torch.float64)
    I_g, I_a = C.random_gravity(3, seed=21, roll_deg=30, pitch_deg=30)
    x = _smooth(3, 3, cam.H, cam.W, seed=4)
    wt = _smooth(3, 3, cam.H, cam.W, seed=9)

    def loss(g, a):
        Hm, y = (GR.inverse_warp if inverse else GR.warp)(cam, x, g, a)
        return (y * wt).sum() + 1e-3 * (Hm * Hm).sum()

    gg, ga = GR.gravity_grads(loss, I_g, I_a, torch.float64)
    h = 1e-6
    for which, base, grad in (("I_g", I_g, gg), ("I_a", I_a, ga)):
        fd = np.zeros_like(grad)
        for i in np.ndindex(base.shape):
            up, dn = base.astype(np.float64).copy(), base.astype(np.float64).copy()
            up[i] += h
            dn[i] -= h
            with torch.no_grad():
                args_up = (torch.tensor(up), torch.tensor(I_a, dtype=torch.float64)) if which == "I_g" else \
                    (torch.tensor(I_g, dtype=torch.float64), torch.tensor(up))
                args_dn = (torch.tensor(dn), torch.tensor(I_a, dtype=torch.float64)) if which == "I_g" else \
                    (torch.tensor(I_g, dtype=torch.float64), torch.tensor(dn))
                fd[i] = (float(loss(*args_up)) - float(loss(*args_dn))) / (2 * h)
        for b in range(base.shape[0]):
            err = np.linalg.norm(grad[b] - fd[b]) / np.linalg.norm(fd[b])
            assert err < 1e-4, (which, b, err, grad[b], fd[b])


@pytest.fixture(scope="module")
def chain_lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("frame_params_grad") / "libframe_params_grad.so")
    # -ffp-contract=off mirrors nvcc -fmad=false
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-mfma", "-o", so,
                    os.path.join(HERE, "harness", "frame_params_grad_host.cpp"), "-lm"], check=True)
    return ctypes.CDLL(so)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


# vidc_frame_params float offsets of the fields the chain reads
OFFSETS = {"H": slice(0, 9), "R": slice(9, 18), "Hinv": slice(18, 27), "px_min": 27, "py_min": 28, "kw": 29, "kh": 30, "ikw": 31,
           "ikh": 32, "w_max": 33, "h_max": 34}


def chain_cases():
    g1, a1 = C.edge_case_gravity()
    g2, a2 = C.random_gravity(24, seed=77, roll_deg=60, pitch_deg=60)     # both sides of the 4:3 branch
    a_gen = np.array([[0.267261, 0.534522, 0.801784], [0.0, 0.8, 0.6]], np.float32)
    g3 = -a_gen                                                           # g = -a with general a: |q| = 0, theta = pi
    g4 = np.array([[0.0, 2.0, 0.0], [0.0, 0.5, 0.0], [1.0, 0.0, 0.0], [-1.0, 0.0, 0.0]], np.float32)   # R = I (ties), +-90 roll
    a4 = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (4, 1))
    return (np.concatenate([g1, g2, g3, g4]).astype(np.float32), np.concatenate([a1, a2, a_gen, a4]).astype(np.float32))


def chain_reference(cam64, I_g, I_a, G, gH, H32):
    """dL/dI_g, dL/dI_a of L = sum_f <G_f, field_f> + <gH, H> by the fp64 restatement's autograd, with the min / max corners
    and the 4:3 branch chosen by the fp32 forward (H32): near +-90 deg of roll two corners differ by an ulp, and fp32 and fp64
    pick different ones."""
    def loss(g, a):
        p = GR.params(cam64, g, a, decide_H=H32)
        L = (p["H"].reshape(-1, 9) * torch.tensor(gH, dtype=torch.float64)).sum()
        for k, sl in OFFSETS.items():
            v = torch.tensor(G[:, sl], dtype=torch.float64)
            L = L + (p[k].reshape(v.shape) * v).sum()
        return L
    return GR.gravity_grads(loss, I_g, I_a, torch.float64)


@pytest.mark.parametrize("cam_name", ["tiny", "S2"])
def test_chain_matches_restatement_autograd(chain_lib, cam_name):
    c = _camera(cam_name)
    cam64 = GR.Camera(c, torch.float64)
    I_g, I_a = chain_cases()
    B = I_g.shape[0]
    rs = np.random.RandomState(3)
    G = np.zeros((B, 48), np.float32)
    for k, sl in OFFSETS.items():
        G[:, sl] = rs.randn(*G[:, sl].shape).astype(np.float32)
    gH = rs.randn(B, 9).astype(np.float32)
    gg = np.zeros((B, 3), np.float32)
    ga = np.zeros((B, 3), np.float32)
    chain_lib.host_frame_params_backward(ctypes.byref(c), _p(I_g), _p(I_a), B, _p(G), _p(gH), _p(gg), _p(ga))
    with torch.no_grad():
        p = GR.params(GR.Camera(c, torch.float32), torch.from_numpy(I_g), torch.from_numpy(I_a))
    rg, ra = chain_reference(cam64, I_g, I_a, G, gH, p["H"])
    # both sides of the branch are exercised
    wide = (p["w_max"] > (4 * p["h_max"]) / 3).numpy()
    assert 0 < wide.sum() < B
    for b in range(B):
        for got, ref in ((gg[b], rg[b]), (ga[b], ra[b])):
            err = np.linalg.norm(got - ref) / max(np.linalg.norm(ref), 1e-30)
            assert err < 1e-5, (cam_name, b, I_g[b], I_a[b], got, ref)


def test_chain_isolates_frames_and_handles_parallel_gravity(chain_lib):
    """|q| = 0 (g parallel to a) passes no gradient through the norm; a NaN frame leaves its neighbours unchanged."""
    c = _camera("S1")
    I_g = np.array([[0.1, 0.9, 0.2], [np.nan, 1.0, 0.0], [0.2, 0.8, -0.1], [0.0, 3.0, 0.0]], np.float32)
    I_a = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (4, 1))
    G = np.random.RandomState(1).randn(4, 48).astype(np.float32)
    out = []
    for rows in ([0, 1, 2, 3], [0], [2], [3]):
        gg = np.zeros((len(rows), 3), np.float32)
        ga = np.zeros_like(gg)
        Ig, Ia, Gr = (np.ascontiguousarray(v[rows]) for v in (I_g, I_a, G))
        chain_lib.host_frame_params_backward(ctypes.byref(c), _p(Ig), _p(Ia), len(rows), _p(Gr), None, _p(gg), _p(ga))
        out.append((gg, ga))
    for j, r in ((1, 0), (2, 2), (3, 3)):
        assert np.array_equal(out[0][0][r], out[j][0][0]) and np.array_equal(out[0][1][r], out[j][1][0])
    assert np.isfinite(out[0][0][3]).all() and np.isfinite(out[0][1][3]).all()
