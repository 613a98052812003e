"""The inverse warp's L2 prefetch box (vidc::inv_prefetch_box, csrc/frame_params.cuh) on the CPU.

A prefetch is a hint, so a wrong box costs only time -- which is why it is checked here: for every frame that passes the
division proof (the only frames the kernel prefetches for) and every 32x32 camera tile, edge tiles included, the box must
hold both bilinear taps of every pixel that reads the canvas.  The taps follow the inverse kernels' coordinate chain
(H, the canvas scale and grid_sample's unnormalisation) evaluated in float64 from the same frame parameters."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import common as C

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def plib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("prefetch_box") / "libprefetch_box.so")
    # -ffp-contract=off mirrors nvcc -fmad=false
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-std=c++17", "-ffp-contract=off", "-mfma", "-o", so,
                    os.path.join(HERE, "harness", "prefetch_box_host.cpp"), "-lm"], check=True)
    return ctypes.CDLL(so)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _gravity(kind):
    if kind == "bench":
        return C.random_gravity(16, seed=1234, roll_deg=30, pitch_deg=30)
    if kind == "roll":
        return C.extreme_roll_gravity(16, seed=5)
    g1, a1 = C.random_gravity(24, seed=5, roll_deg=90, pitch_deg=85)      # includes frames whose horizon crosses the image
    g2, a2 = C.edge_case_gravity()
    return np.concatenate([g1, g2]), np.concatenate([a1, a2])


@pytest.mark.parametrize("cam_name,kind", [("S2", "bench"), ("S3", "roll"), ("S1", "wide"), ("tiny", "wide"), ("S2", "wide")])
def test_inverse_prefetch_box_holds_every_tap(plib, cam_name, kind):
    from vi_depth_completion_b200._cabi import VidcCamera, lib
    cam = C.CAMERAS[cam_name]
    c = VidcCamera()
    assert lib().vidc_camera_init(*[float(v) for v in cam], ctypes.byref(c)) == 0
    I_g, I_a = (np.ascontiguousarray(x, dtype=np.float32) for x in _gravity(kind))
    B, W, H = I_g.shape[0], c.W, c.H
    tx, ty = (W + 31) // 32, (H + 31) // 32
    boxes = np.zeros((B, ty, tx, 4), np.int32)
    proven = np.zeros(B, np.uint8)
    prm = np.zeros((B, 48), np.float32)
    plib.host_inv_prefetch_boxes(ctypes.byref(c), _p(I_g), _p(I_a), B, _p(boxes), _p(proven), _p(prm))
    X, Y = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    n_tiles = 0
    for b in np.nonzero(proven)[0]:
        Hm, (px_min, py_min, kw, kh) = prm[b, :9].astype(np.float64), prm[b, 27:31].astype(np.float64)
        s = Hm[6] * X + Hm[7] * Y + Hm[8]
        gx = c.inv_half_w * (kw * ((Hm[0] * X + Hm[1] * Y + Hm[2]) / s - px_min) - c.cx)     # :245 and grid_sample's
        gy = c.inv_half_h * (kh * ((Hm[3] * X + Hm[4] * Y + Hm[5]) / s - py_min) - c.cy)     # unnormalisation
        x0, y0 = np.floor(((gx + 1) * W - 1) / 2), np.floor(((gy + 1) * H - 1) / 2)
        for j in range(ty):
            for i in range(tx):
                sl = (slice(32 * j, 32 * j + 32), slice(32 * i, 32 * i + 32))
                xs, ys = x0[sl], y0[sl]
                assert np.isfinite(xs).all() and np.isfinite(ys).all()
                bx0, by0, bx1, by1 = boxes[b, j, i]
                # taps x0, x0 + 1 (and y0, y0 + 1) that fall inside the canvas: those the kernel reads
                for dx in (0, 1):
                    for dy in (0, 1):
                        tx_, ty_ = xs + dx, ys + dy
                        live = (tx_ >= 0) & (tx_ <= W - 1) & (ty_ >= 0) & (ty_ <= H - 1)
                        outside = live & ~((tx_ >= bx0) & (tx_ <= bx1) & (ty_ >= by0) & (ty_ <= by1))
                        assert not outside.any(), f"{cam_name}/{kind} frame {b} tile ({i},{j}): tap outside {boxes[b, j, i]}"
                n_tiles += 1
    assert n_tiles >= 8 * tx * ty                                     # most frames are prefetched for
    if kind == "wide":                                                # and some are not: the kernel skips them
        assert not proven.all()
