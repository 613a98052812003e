"""warp_rgbd_u8: the fused forward warp on (B,h,w,3) uint8 frames gives the bits of warp_rgbd(to_tensor_u8(frames), ...).

Every output is compared bit for bit (Cg_H_C, RGB, depth, mask, coverage) with the composition of the two existing entry
points, over the compile-time canvases, S3's rolls (whose tiles run lanes along Y), the runtime-geometry canvases, inputs
smaller and larger than the canvas, both depth modes and none, with and without mask and coverage, the params= and the
I_g / I_a forms, the torch operators and the C ABI, B = 1 and 256, frames one byte off alignment and a NaN-gravity frame.

The switches are read once per process, so each setting runs the cases in a fresh process with VIDC_* stripped from the
inherited environment.  That process also records which kernels each uint8 call launches (as tests/test_gpu_dispatch.py
does), compared with a table frozen from a run on a B200: `python tests/test_gpu_warp_u8.py --freeze` prints it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SETTINGS = {"default": {}, "shear0": {"VIDC_SHEAR": "0"}, "tma": {"VIDC_TMA": "1"}, "tma_store0": {"VIDC_TMA_STORE": "0"},
            "pf_bulk0": {"VIDC_PF_BULK": "0"}, "tile_skip0": {"VIDC_TILE_SKIP": "0"}}

CANVASES = {"S1": (202.0, 202.0, 159.93827, 119.938015), "S2": (404.0, 404.0, 319.87654, 239.87603),
            "640x489": (404.0, 404.0, 319.87654, 244.4), "S3": (577.87061, 580.25851, 319.87654, 239.87603),
            "416x301": (300.0, 300.0, 207.7, 150.2), "300x201": (250.0, 250.0, 149.7, 100.2)}


def _frames(B, h, w, seed):
    """(B,h,w,3) uint8; frame 0 holds every byte value (a ramp), the others are random."""
    rs = np.random.RandomState(seed)
    u8 = rs.randint(0, 256, size=(B, h, w, 3)).astype(np.uint8)
    u8[0] = (np.arange(h * w * 3) % 256).astype(np.uint8).reshape(h, w, 3)
    return u8


def _child():
    import ctypes

    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    from tests import common as C
    from vi_depth_completion_b200._cabi import VIDC_BILINEAR, VIDC_NEAREST, check, lib
    from vi_depth_completion_b200.gravity import to_tensor_u8
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment, _image, _stream_ptr

    dev = torch.device("cuda", 0)
    bits, kernels = {}, {}

    def record(fn):
        torch.cuda.synchronize()
        n0 = lib().vidc_launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        n = lib().vidc_launch_count() - n0
        names = []
        for e in sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start):
            if e.name.startswith("Memset"):
                names.append("memset")
            elif not e.name.startswith("Memcpy") and "at::" not in e.name:
                names.append(e.name.split("(")[0].removeprefix("void ").removeprefix("vidc_k::").strip())
        return out, f"{n}: " + " + ".join(names)

    def differing_bits(got, want):
        n = 0
        for x, y in zip(got, want):
            if x is None or y is None:
                n += 0 if x is None and y is None else 1 << 30
                continue
            x, y = x.contiguous(), y.contiguous()
            if x.shape != y.shape or x.dtype != y.dtype:
                n += 1 << 30
                continue
            if x.dtype == torch.float32:
                x, y = x.view(torch.int32), y.view(torch.int32)
            n += int((x != y).sum())
        return n

    def cabi(w, u8, depth, g, a, mode, params=None, mask=True, coverage=True, fn=None):
        """vidc_warp_rgbd_u8 (fn=None) or vidc_warp_rgbd on the float frames, straight through the C ABI"""
        B, Hc, Wc = u8.shape[0], int(w.H), int(w.W)
        rgb_w = torch.empty(B, 3, Hc, Wc, device=dev)
        dw = torch.empty(B, 1, Hc, Wc, device=dev) if depth is not None else None
        m = torch.empty(B, 1, Hc, Wc, dtype=torch.uint8, device=dev) if mask else None
        cov = torch.empty(B, dtype=torch.int32, device=dev) if coverage else None
        Hm = torch.empty(B, 3, 3, device=dev) if params is None else None
        ws = w._params_ws(B, dev) if params is None else params.ws
        di, dwi, rwi = (ctypes.byref(_image(depth)) if depth is not None else None), (ctypes.byref(_image(dw)) if dw is not None else None), \
            ctypes.byref(_image(rgb_w))
        gp, ap = (g.data_ptr(), a.data_ptr()) if params is None else (None, None)
        tail = (ws.data_ptr(), Hm.data_ptr() if Hm is not None else None, rwi, dwi, m.data_ptr() if mask else None,
                cov.data_ptr() if coverage else None, _stream_ptr(dev))
        if fn is None:
            check(lib().vidc_warp_rgbd_u8(ctypes.byref(w._cam), u8.data_ptr(), B, u8.shape[1], u8.shape[2], di, gp, ap, B, mode, *tail))
        else:
            check(lib().vidc_warp_rgbd(ctypes.byref(w._cam), ctypes.byref(_image(fn)), di, gp, ap, B, mode, *tail))
        return Hm, rgb_w, dw, m, cov

    def case(name, w, u8, depth, g, a, depth_mode="bilinear", mask=True, coverage=False, params=None, front="python"):
        x = to_tensor_u8(u8)
        mode = VIDC_BILINEAR if depth_mode == "bilinear" else VIDC_NEAREST
        if front == "cabi":
            got, kernels[name] = record(lambda: cabi(w, u8, depth, g, a, mode, params, mask, coverage))
            want = cabi(w, u8, depth, g, a, mode, params, mask, coverage, fn=x)
        else:
            kw = dict(depth_mode=depth_mode, with_mask=mask, with_coverage=coverage, params=params)
            ga = (None, None) if params is not None else (g, a)
            got, kernels[name] = record(lambda: w.warp_rgbd_u8(u8, depth, *ga, **kw))
            want = w.warp_rgbd(x, depth, *ga, **kw)
            assert got[1].is_contiguous() and got[1].dtype == torch.float32
        torch.cuda.synchronize()
        bits[name] = differing_bits(got, want)
        return got

    rolls = {"S3": C.extreme_roll_gravity(7, seed=31)}
    with torch.no_grad():
        for canvas, intr in CANVASES.items():
            w = Warping2DOFAlignment(*intr)
            Hc, Wc = int(w.H), int(w.W)
            I_g, I_a = rolls.get(canvas, C.random_gravity(3, seed=11, roll_deg=30, pitch_deg=30))
            B = I_g.shape[0]
            g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)
            u8 = torch.from_numpy(_frames(B, Hc, Wc, seed=5)).to(dev)
            depth = torch.from_numpy(np.random.RandomState(6).rand(B, 1, Hc, Wc).astype(np.float32) * 9 + 0.5).to(dev)
            if not kernels:
                record(lambda: w.warp_rgbd_u8(u8, depth, g, a))          # first profiler session of the process: not recorded
            p = w.prepare(g, a)
            case(f"{canvas}/op", w, u8, depth, g, a)
            case(f"{canvas}/op/nearest", w, u8, depth, g, a, depth_mode="nearest")
            case(f"{canvas}/op/params", w, u8, depth, g, a, params=p)
            case(f"{canvas}/no_depth", w, u8, None, g, a)
            case(f"{canvas}/coverage", w, u8, depth, g, a, coverage=True)
            case(f"{canvas}/coverage/no_mask", w, u8, depth, g, a, mask=False, coverage=True, depth_mode="nearest")
            case(f"{canvas}/cabi", w, u8, depth, g, a, coverage=True, front="cabi")
            case(f"{canvas}/cabi/params/no_depth", w, u8, None, g, a, params=p, front="cabi")
            case(f"{canvas}/cabi/nearest/no_mask", w, u8, depth, g, a, depth_mode="nearest", mask=False, front="cabi")
            if canvas == "S1":                                        # ToTensor done by torch itself
                got = w.warp_rgbd_u8(u8, depth, g, a)
                want = w.warp_rgbd(u8.cpu().permute(0, 3, 1, 2).float().div(255).to(dev), depth, g, a)
                bits["S1/torch_to_tensor"] = differing_bits(got, want)
            if canvas != "S2":
                continue
            for tag, (h, wd) in {"smaller": (360, 480), "larger": (600, 800)}.items():
                su8 = torch.from_numpy(_frames(B, h, wd, seed=7)).to(dev)
                sd = torch.from_numpy(np.random.RandomState(8).rand(B, 1, h, wd).astype(np.float32) + 1).to(dev)
                case(f"S2/{tag}/op", w, su8, sd, g, a)
                case(f"S2/{tag}/no_depth", w, su8, None, g, a)
                case(f"S2/{tag}/cabi", w, su8, sd, g, a, coverage=True, front="cabi")
            case("S2/depth3d", w, u8, depth[:, 0], g, a)
            buf = torch.empty(u8.numel() + 16, dtype=torch.uint8, device=dev)
            off = buf[1:1 + u8.numel()].view(u8.shape)                # data pointer one byte past a 16-byte boundary
            off.copy_(u8)
            case("S2/offset1/op", w, off, depth, g, a)
            case("S2/offset1/cabi", w, off, depth, g, a, coverage=True, front="cabi")
            case("S2/B1", w, u8[:1], depth[:1], g[:1], a[:1])
            I_g256, I_a256 = C.random_gravity(256, seed=12, roll_deg=30, pitch_deg=30)
            g256, a256 = torch.from_numpy(I_g256).to(dev), torch.from_numpy(I_a256).to(dev)
            u256 = torch.from_numpy(_frames(256, Hc, Wc, seed=9)).to(dev)
            d256 = torch.from_numpy(np.random.RandomState(10).rand(256, 1, Hc, Wc).astype(np.float32) + 1).to(dev)
            case("S2/B256", w, u256, d256, g256, a256)
            case("S2/B256/coverage", w, u256, d256, g256, a256, coverage=True)
            # a NaN-gravity frame among finite ones: zeros there, its neighbours as without it
            gn = g.clone()
            gn[1, 0] = float("nan")
            got = case("S2/nan_gravity", w, u8, depth, gn, a, coverage=True)
            keep = torch.tensor([0, 2], device=dev)
            alone = w.warp_rgbd_u8(u8[keep], depth[keep], g[keep], a[keep], with_coverage=True)
            iso = differing_bits([o[keep] for o in got[1:]], list(alone[1:]))
            iso += int((got[1][1] != 0).sum() + (got[2][1] != 0).sum() + (got[3][1] != 0).sum() + (got[4][1] != 0).sum())
            bits["S2/nan_gravity/isolated"] = iso
    print(json.dumps({"bits": bits, "kernels": kernels}), flush=True)


def _run(setting):
    env = {k: v for k, v in os.environ.items() if not k.startswith("VIDC_")}
    env.update(SETTINGS[setting])
    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=1200)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])


def _expected(setting):
    want = dict(DEFAULT)
    want.update(DIFFERS.get(setting, {}))
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_u8_warp_matches_to_tensor_then_warp(cuda_device, setting):
    got = _run(setting)
    bad = {k: v for k, v in got["bits"].items() if v != 0}
    assert not bad, f"{setting}: differing bits per case: {bad}"
    want = _expected(setting)
    assert set(got["kernels"]) == set(want), f"calls differ: {sorted(set(got['kernels']) ^ set(want))}"
    wrong = [f"{k}\n    want {want[k]}\n    got  {got['kernels'][k]}" for k in sorted(want) if got["kernels"][k] != want[k]]
    assert not wrong, f"{setting}: {len(wrong)} calls launch other kernels:\n" + "\n".join(wrong)


@pytest.mark.gpu
def test_u8_warp_errors_and_autograd(cuda_device):
    import torch

    from vi_depth_completion_b200.gravity import to_tensor_u8
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    from tests import common as C

    w = Warping2DOFAlignment(*CANVASES["S1"])
    I_g, I_a = C.random_gravity(2, seed=3)
    g, a = torch.from_numpy(I_g).to(cuda_device), torch.from_numpy(I_a).to(cuda_device)
    u8 = torch.from_numpy(_frames(2, 240, 320, seed=4)).to(cuda_device)
    depth = torch.rand(2, 1, 240, 320, device=cuda_device) + 1
    with pytest.raises(RuntimeError):
        w.warp_rgbd_u8(u8.float(), depth, g, a)                             # float frames
    with pytest.raises(RuntimeError):
        w.warp_rgbd_u8(torch.zeros(2, 240, 320, 4, dtype=torch.uint8, device=cuda_device), depth, g, a)   # C = 4
    with pytest.raises(RuntimeError):
        w.warp_rgbd_u8(u8.cpu(), depth, g, a)                               # host frames
    with pytest.raises(RuntimeError):
        w.warp_rgbd_u8(u8, depth.cpu(), g, a)                               # depth on another device
    with pytest.raises(RuntimeError):
        w.warp_rgbd_u8(u8, depth.cpu(), g, a, with_coverage=True)           # the same through the C ABI
    with pytest.raises(AssertionError):
        w.warp_rgbd_u8(u8, depth, g[:1], a[:1])                             # batch mismatch, torch operator
    with pytest.raises(AssertionError):
        w.warp_rgbd_u8(u8, depth, g[:1], a[:1], with_coverage=True)         # batch mismatch, C ABI
    with pytest.raises(AssertionError):
        w.warp_rgbd_u8(u8, depth, params=w.prepare(g[:1], a[:1]))
    with pytest.raises(RuntimeError):
        w.warp_rgbd(u8, depth, g, a)                                        # warp_rgbd keeps rejecting uint8
    # a non-contiguous view of the frames is made contiguous
    view = u8.permute(0, 3, 1, 2).contiguous().permute(0, 2, 3, 1)
    assert not view.is_contiguous()
    got, want = w.warp_rgbd_u8(view, depth, g, a), w.warp_rgbd(to_tensor_u8(u8), depth, g, a)
    assert all(torch.equal(x, y) for x, y in zip(got, want))
    # forward-only: depth that requires grad, and gravity that requires grad
    d = depth.clone().requires_grad_(True)
    out = w.warp_rgbd_u8(u8, d, g, a)
    assert out[2].requires_grad
    with pytest.raises(NotImplementedError):
        out[2].sum().backward()
    gg = g.clone().requires_grad_(True)
    for kw in ({}, {"with_coverage": True}):
        out = w.warp_rgbd_u8(u8, depth, gg, a, **kw)
        with pytest.raises(NotImplementedError):
            out[1].sum().backward()
    p = w.prepare(gg, a)
    with pytest.raises(NotImplementedError):
        w.warp_rgbd_u8(u8, depth, params=p)[1].sum().backward()


@pytest.mark.gpu
def test_u8_operators_trace_under_torch_compile(cuda_device):
    import torch

    from vi_depth_completion_b200 import _torchops
    ops = _torchops.ops()
    assert ops is not None
    intr = CANVASES["S1"]
    u8 = torch.from_numpy(_frames(2, 240, 320, seed=4)).to(cuda_device)
    depth = torch.rand(2, 1, 240, 320, device=cuda_device) + 1
    g = torch.tensor([[0.1, 0.99, 0.05], [-0.2, 0.97, 0.1]], device=cuda_device)
    a = torch.tensor([[0.0, 1.0, 0.0]] * 2, device=cuda_device)

    def f(u8, depth, g, a):
        ws, _ = ops.frame_params(g, a, *intr)
        return ops.warp_rgbd_u8(u8, depth, g, a, *intr, 0)[1] + ops.warp_rgbd_u8_prepared(u8, depth, ws, *intr, 0)[0]

    got = torch.compile(f, fullgraph=True, backend="eager")(u8, depth, g, a)
    assert torch.equal(got, f(u8, depth, g, a))


def _freeze():
    runs = {s: _run(s) for s in SETTINGS}
    for s, r in runs.items():
        print(f"# {s}: cases with differing bits: {({k: v for k, v in r['bits'].items() if v}) or 'none'} of {len(r['bits'])}")
    tables = {s: r["kernels"] for s, r in runs.items()}
    base = tables["default"]
    print("DEFAULT = {")
    for k, v in base.items():
        print(f"    {k!r}: {v!r},")
    print("}")
    print("DIFFERS = {")
    for s, t in tables.items():
        if s != "default":
            print(f"    {s!r}: {{")
            for k, v in t.items():
                if v != base[k]:
                    print(f"        {k!r}: {v!r},")
            print("    },")
    print("}")


# frozen from a run on a B200 (NVIDIA B200, 1000 W)
DEFAULT = {
    'S1/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S1/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S1/op/params': '1: warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S1/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, false, true>',
    'S1/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S1/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S1/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S1/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<320, 240, false, true>',
    'S1/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
    'S2/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/op/params': '1: warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, false, true>',
    'S2/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<640, 480, false, true>',
    'S2/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/smaller/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    'S2/smaller/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
    'S2/smaller/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    'S2/larger/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    'S2/larger/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
    'S2/larger/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    'S2/depth3d': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/offset1/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/offset1/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/B1': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/B256': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/B256/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S2/nan_gravity': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    '640x489/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    '640x489/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    '640x489/op/params': '1: warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    '640x489/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, false, true>',
    '640x489/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    '640x489/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    '640x489/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    '640x489/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<640, 489, false, true>',
    '640x489/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
    'S3/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S3/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S3/op/params': '1: warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S3/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, false, true>',
    'S3/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S3/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S3/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    'S3/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<640, 480, false, true>',
    'S3/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
    '416x301/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '416x301/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '416x301/op/params': '1: warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '416x301/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, false, true>',
    '416x301/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '416x301/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '416x301/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '416x301/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<0, 0, false, true>',
    '416x301/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
    '300x201/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    '300x201/op/nearest': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    '300x201/op/params': '1: warp_forward_u8_kernel<true>',
    '300x201/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
    '300x201/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    '300x201/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    '300x201/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    '300x201/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
    '300x201/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
}
DIFFERS = {
    'shear0': {
        'S1/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S1/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S1/op/params': '1: warp_forward_u8_kernel<true>',
        'S1/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S1/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S1/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S1/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S1/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        'S1/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/op/params': '1: warp_forward_u8_kernel<true>',
        'S2/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S2/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        'S2/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/smaller/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/smaller/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S2/smaller/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/larger/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/larger/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S2/larger/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/depth3d': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/offset1/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/offset1/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/B1': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/B256': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/B256/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/nan_gravity': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '640x489/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '640x489/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '640x489/op/params': '1: warp_forward_u8_kernel<true>',
        '640x489/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        '640x489/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '640x489/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '640x489/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '640x489/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        '640x489/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S3/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S3/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S3/op/params': '1: warp_forward_u8_kernel<true>',
        'S3/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S3/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S3/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S3/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S3/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        'S3/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '416x301/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '416x301/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '416x301/op/params': '1: warp_forward_u8_kernel<true>',
        '416x301/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        '416x301/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '416x301/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '416x301/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '416x301/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        '416x301/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        '300x201/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
    },
    'tma': {
        'S1/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S1/op/nearest': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S1/op/params': '1: warp_forward_u8_kernel<true>',
        'S1/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
        'S1/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S1/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S1/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S1/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        'S1/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/op/nearest': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/op/params': '1: warp_forward_u8_kernel<true>',
        'S2/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
        'S2/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        'S2/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/depth3d': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/offset1/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/offset1/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/B1': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/B256': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/B256/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S2/nan_gravity': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '640x489/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '640x489/op/nearest': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '640x489/op/params': '1: warp_forward_u8_kernel<true>',
        '640x489/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
        '640x489/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '640x489/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '640x489/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '640x489/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        '640x489/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S3/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S3/op/nearest': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S3/op/params': '1: warp_forward_u8_kernel<true>',
        'S3/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
        'S3/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S3/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S3/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        'S3/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        'S3/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '416x301/op': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '416x301/op/nearest': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '416x301/op/params': '1: warp_forward_u8_kernel<true>',
        '416x301/no_depth': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<false>',
        '416x301/coverage': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '416x301/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '416x301/cabi': '2: memset + frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
        '416x301/cabi/params/no_depth': '1: warp_forward_u8_kernel<false>',
        '416x301/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_forward_u8_kernel<true>',
    },
    'tma_store0': {
        'S1/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S1/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S1/op/params': '1: warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S1/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, false, false>',
        'S1/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S1/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S1/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S1/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<320, 240, false, false>',
        'S1/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, false>',
        'S2/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/op/params': '1: warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, false, false>',
        'S2/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<640, 480, false, false>',
        'S2/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/depth3d': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/offset1/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/offset1/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/B1': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/B256': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/B256/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S2/nan_gravity': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        '640x489/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        '640x489/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        '640x489/op/params': '1: warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        '640x489/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, false, false>',
        '640x489/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        '640x489/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        '640x489/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        '640x489/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<640, 489, false, false>',
        '640x489/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, false>',
        'S3/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S3/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S3/op/params': '1: warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S3/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, false, false>',
        'S3/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S3/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S3/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        'S3/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<640, 480, false, false>',
        'S3/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, false>',
        '416x301/op': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, false>',
        '416x301/op/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, false>',
        '416x301/op/params': '1: warp_rgbd_shear_u8_kernel<0, 0, true, false>',
        '416x301/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, false, false>',
        '416x301/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, false>',
        '416x301/coverage/no_mask': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, false>',
        '416x301/cabi': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, false>',
        '416x301/cabi/params/no_depth': '1: warp_rgbd_shear_u8_kernel<0, 0, false, false>',
        '416x301/cabi/nearest/no_mask': '2: frame_params_tiles_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, false>',
    },
    'pf_bulk0': {
    },
    'tile_skip0': {
        'S1/op': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
        'S1/op/nearest': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
        'S1/no_depth': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, false, true>',
        'S1/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
        'S1/coverage/no_mask': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
        'S1/cabi': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
        'S1/cabi/nearest/no_mask': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<320, 240, true, true>',
        'S2/op': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/op/nearest': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/no_depth': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, false, true>',
        'S2/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/coverage/no_mask': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/cabi': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/cabi/nearest/no_mask': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/smaller/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/smaller/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S2/smaller/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/larger/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/larger/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        'S2/larger/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        'S2/depth3d': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/offset1/op': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/offset1/cabi': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/B1': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/B256': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/B256/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S2/nan_gravity': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        '640x489/op': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
        '640x489/op/nearest': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
        '640x489/no_depth': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, false, true>',
        '640x489/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
        '640x489/coverage/no_mask': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
        '640x489/cabi': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
        '640x489/cabi/nearest/no_mask': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 489, true, true>',
        'S3/op': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S3/op/nearest': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S3/no_depth': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, false, true>',
        'S3/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S3/coverage/no_mask': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S3/cabi': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        'S3/cabi/nearest/no_mask': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<640, 480, true, true>',
        '416x301/op': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
        '416x301/op/nearest': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
        '416x301/no_depth': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, false, true>',
        '416x301/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
        '416x301/coverage/no_mask': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
        '416x301/cabi': '2: memset + frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
        '416x301/cabi/nearest/no_mask': '2: frame_params_kernel + warp_rgbd_shear_u8_kernel<0, 0, true, true>',
        '300x201/op': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/op/nearest': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/no_depth': '2: frame_params_kernel + warp_forward_u8_kernel<false>',
        '300x201/coverage': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/coverage/no_mask': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/cabi': '2: memset + frame_params_kernel + warp_forward_u8_kernel<true>',
        '300x201/cabi/nearest/no_mask': '2: frame_params_kernel + warp_forward_u8_kernel<true>',
    },
}


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    if "--child" in sys.argv:
        _child()
    elif "--freeze" in sys.argv:
        _freeze()
