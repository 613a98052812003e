"""Which kernels each warp entry point launches, for every environment switch and the inputs that steer the choice.

Every kernel family gives the same bits, so a call that silently falls from the sheared kernel to the straight-row one, or
loses its TMA write-out, passes every parity and golden test and only loses throughput.  This test pins the choice: for each
call it records the kernels the call launches (demangled names with their template arguments, in launch order, memsets as
"memset") and how far vidc_launch_count() moves, and compares them with a table frozen from a run on a B200.

The switches are read once per process, so each setting runs the calls in a fresh process with VIDC_* stripped from the
inherited environment.  `python tests/test_gpu_dispatch.py --freeze` prints the table for the current build."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SETTINGS = {"default": {}, "shear0": {"VIDC_SHEAR": "0"}, "shear1": {"VIDC_SHEAR": "1"}, "tma": {"VIDC_TMA": "1"},
            "inv_box": {"VIDC_INV_BOX": "1"}, "tma_store0": {"VIDC_TMA_STORE": "0"}, "tile_skip0": {"VIDC_TILE_SKIP": "0"}}

# (name, intrinsics): the three compile-time canvases, a runtime canvas whose width is a multiple of 32, and one whose width
# is not (300x201)
CANVASES = [("S2", (404.0, 404.0, 319.87654, 239.87603)), ("S1", (202.0, 202.0, 159.93827, 119.938015)),
            ("640x489", (404.0, 404.0, 319.87654, 244.4)), ("416x301", (300.0, 300.0, 207.7, 150.2)),
            ("300x201", (250.0, 250.0, 149.7, 100.2))]
B = 2


def _child():
    import ctypes

    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    from tests import common as C
    from vi_depth_completion_b200 import _cabi
    from vi_depth_completion_b200._cabi import check, lib
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment, _image, _stream_ptr

    dev = torch.device("cuda", 0)
    gen = torch.Generator(device=dev).manual_seed(5)
    rand = lambda *s: torch.rand(*s, device=dev, generator=gen)

    def offset(t):                                   # same shape, data pointer one float past a 16-byte boundary
        buf = torch.empty(t.numel() + 4, device=dev)
        v = buf[1:1 + t.numel()].view(t.shape)
        v.copy_(t)
        return v

    def strided(t, pad=64):                          # a view whose rows are longer than its width
        big = torch.zeros(*t.shape[:-1], t.shape[-1] + pad, device=dev)
        big[..., :t.shape[-1]] = t
        return big[..., :t.shape[-1]]

    def record(fn):
        torch.cuda.synchronize()
        n0 = lib().vidc_launch_count()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        n = lib().vidc_launch_count() - n0
        names = []
        for e in sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start):
            if e.name.startswith("Memset"):
                names.append("memset")
            elif not e.name.startswith("Memcpy") and "at::" not in e.name:
                names.append(e.name.split("(")[0].removeprefix("void ").removeprefix("vidc_k::").strip())
        return f"{n}: " + " + ".join(names)

    table = {}
    for canvas, intr in CANVASES:
        w = Warping2DOFAlignment(*intr)
        Hc, Wc = int(w.H), int(w.W)
        I_g, I_a = C.random_gravity(B, seed=1234, roll_deg=30, pitch_deg=30)
        g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)
        rgb, depth, nrm = rand(B, 3, Hc, Wc), rand(B, 1, Hc, Wc) * 9 + 0.5, rand(B, 3, Hc, Wc) - 0.5
        x1, x2, x5 = rand(B, 1, Hc, Wc), rand(B, 2, Hc, Wc), rand(B, 5, Hc, Wc)
        rgb_cl, nrm_cl = rgb.contiguous(memory_format=torch.channels_last), nrm.contiguous(memory_format=torch.channels_last)
        N = 16
        tracks = torch.zeros(B, N, 4, dtype=torch.float64, device=dev)
        tracks[..., 0] = torch.arange(N, device=dev)
        tracks[..., 1:3] = (rand(B, N, 2).double() - 0.5)
        tracks[..., 3] = rand(B, N).double() * 4 + 1
        counts = torch.full((B,), N, dtype=torch.int32, device=dev)
        fc, cc = (intr[0], intr[1]), (intr[2], intr[3])
        held = {}

        def prepare():
            held["p"] = w.prepare(g, a)

        calls = [
            ("warp_rgbd", lambda: w.warp_rgbd(rgb, depth, g, a)),
            ("warp_rgbd/no_depth", lambda: w.warp_rgbd(rgb, None, g, a)),
            ("warp_rgbd/coverage", lambda: w.warp_rgbd(rgb, depth, g, a, with_coverage=True)),
            ("warp_rgbd/nearest", lambda: w.warp_rgbd(rgb, depth, g, a, depth_mode="nearest")),
            ("prepare", prepare),
            ("warp_rgbd/params", lambda: w.warp_rgbd(rgb, depth, params=held["p"])),
            ("warp_rgb_sparse_depth", lambda: w.warp_rgb_sparse_depth(rgb, tracks, counts, fc, cc, g, a)),
            ("forward/C1", lambda: w.warp_with_gravity_center_aligned(x1, g, a)),
            ("forward/C2", lambda: w.warp_with_gravity_center_aligned(x2, g, a)),
            ("forward/C3", lambda: w.warp_with_gravity_center_aligned(rgb, g, a)),
            ("forward/C5", lambda: w.warp_with_gravity_center_aligned(x5, g, a)),            # channel groups 4 + 1
            ("forward/C3/nearest", lambda: w.warp_with_gravity_center_aligned(rgb, g, a, interp_mode="nearest")),
            ("forward/C3/bicubic", lambda: w.warp_with_gravity_center_aligned(rgb, g, a, interp_mode="bicubic")),
            ("unwarp_normals", lambda: w.unwarp_normals(nrm, g, a)),
            ("unwarp_normals/raw", lambda: w.unwarp_normals(nrm, g, a, normalize=False)),
            ("unwarp_normals/valid", lambda: w.unwarp_normals(nrm, g, a, with_valid=True)),
            ("unwarp_normals/raw_valid", lambda: w.unwarp_normals(nrm, g, a, normalize=False, with_valid=True)),
            ("unwarp_normals/params", lambda: w.unwarp_normals(nrm, params=held["p"])),
            ("inverse_warp_normal_image", lambda: w.inverse_warp_normal_image_with_gravity_center_aligned(nrm, g, a)),
            ("channels_last/forward", lambda: w.warp_with_gravity_center_aligned(rgb_cl, g, a)),
            ("channels_last/warp_rgbd", lambda: w.warp_rgbd(rgb_cl, depth, g, a)),
            ("channels_last/unwarp_normals", lambda: w.unwarp_normals(nrm_cl, g, a)),
            ("channels_last/unwarp_normals/raw", lambda: w.unwarp_normals(nrm_cl, g, a, normalize=False)),
        ]
        if canvas == "S2":
            small_rgb, small_dep = rand(B, 3, 360, 480), rand(B, 1, 360, 480) + 1
            s_rgb, s_dep, s_nrm = strided(rgb), strided(depth), strided(nrm)
            o_rgb, o_dep, o_nrm = offset(rgb), offset(depth), offset(nrm)
            packed = torch.cat([rgb, depth], 1).contiguous(memory_format=torch.channels_last)
            cam, st = ctypes.byref(w._cam), _stream_ptr(dev)
            ws, Hout = w._params_ws(B, dev), torch.empty(B, 3, 3, device=dev)
            out3, out1 = offset(torch.empty(B, 3, Hc, Wc, device=dev)), offset(torch.empty(B, 1, Hc, Wc, device=dev))
            mask = torch.empty(B, 1, Hc, Wc, dtype=torch.uint8, device=dev)
            rgb_out = torch.empty(B, 3, Hc, Wc, device=dev)
            im = lambda t: ctypes.byref(_image(t))
            calls += [
                ("warp_normal_image", lambda: w.warp_normal_image_with_gravity_center_aligned(nrm, g, a)),
                ("warp_with_homography", lambda: w.warp_with_homography(rgb, held["p"].H)),
                ("warp_rgbd_packed", lambda: w.warp_rgbd_packed(packed, g, a)),
                ("smaller_input/warp_rgbd", lambda: w.warp_rgbd(small_rgb, small_dep, g, a)),
                ("smaller_input/forward/C3", lambda: w.warp_with_gravity_center_aligned(small_rgb, g, a)),
                ("strided/warp_rgbd", lambda: w.warp_rgbd(s_rgb, s_dep, g, a)),
                ("strided/forward/C3", lambda: w.warp_with_gravity_center_aligned(s_rgb, g, a)),
                ("strided/unwarp_normals", lambda: w.unwarp_normals(s_nrm, g, a)),
                ("offset_in/warp_rgbd", lambda: w.warp_rgbd(o_rgb, o_dep, g, a)),
                ("offset_in/forward/C3", lambda: w.warp_with_gravity_center_aligned(o_rgb, g, a)),
                ("offset_in/unwarp_normals", lambda: w.unwarp_normals(o_nrm, g, a)),
                ("offset_in/warp_rgb_sparse_depth", lambda: w.warp_rgb_sparse_depth(o_rgb, tracks, counts, fc, cc, g, a)),
                ("offset_out/warp_rgbd", lambda: check(lib().vidc_warp_rgbd(
                    cam, im(rgb), im(depth), g.data_ptr(), a.data_ptr(), B, _cabi.VIDC_BILINEAR, ws.data_ptr(), Hout.data_ptr(),
                    im(out3), im(out1), mask.data_ptr(), None, st))),
                ("offset_out/forward/C3", lambda: check(lib().vidc_warp_forward(
                    cam, im(rgb), g.data_ptr(), a.data_ptr(), B, _cabi.VIDC_BILINEAR, ws.data_ptr(), Hout.data_ptr(), im(out3), st))),
                ("offset_out/unwarp_normals", lambda: check(lib().vidc_unwarp_normals(
                    cam, im(nrm), g.data_ptr(), a.data_ptr(), B, 1, ws.data_ptr(), Hout.data_ptr(), im(out3), None, st))),
                ("offset_out/warp_rgb_sparse_depth", lambda: check(lib().vidc_warp_rgb_sparse_depth(
                    cam, im(rgb), tracks.data_ptr(), counts.data_ptr(), N, 4, fc[0], fc[1], cc[0], cc[1], g.data_ptr(), a.data_ptr(),
                    B, _cabi.VIDC_BILINEAR, ws.data_ptr(), Hout.data_ptr(), im(rgb_out), im(out1),
                    mask.data_ptr(), None, st))),
            ]
        with torch.no_grad():
            if not table:
                record(calls[0][1])                  # first profiler session of the process: warm-up, not recorded
            for name, fn in calls:
                table[f"{canvas}/{name}"] = record(fn)
    print(json.dumps(table), flush=True)


def _run(setting):
    env = {k: v for k, v in os.environ.items() if not k.startswith("VIDC_")}
    env.update(SETTINGS[setting])
    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child"], cwd=ROOT, env=env, capture_output=True, text=True,
                         timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])


def _expected(setting):
    want = dict(DEFAULT)
    want.update(DIFFERS.get(setting, {}))
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_each_call_reaches_its_kernels(cuda_device, setting):
    got, want = _run(setting), _expected(setting)
    assert set(got) == set(want), f"calls differ: {sorted(set(got) ^ set(want))}"
    bad = [f"{k}\n    want {want[k]}\n    got  {got[k]}" for k in sorted(want) if got[k] != want[k]]
    assert not bad, f"{setting}: {len(bad)} calls launch other kernels:\n" + "\n".join(bad)


def _freeze():
    tables = {s: _run(s) for s in SETTINGS}
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


# ---- frozen from a run on a B200, before the kernel-selection decisions of vidc_kernels.cu were each written once -----------
DEFAULT = {
    'S2/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
    'S2/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, false, true>',
    'S2/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
    'S2/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
    'S2/prepare': '1: frame_params_tiles_kernel',
    'S2/warp_rgbd/params': '1: warp_rgbd_shear_kernel<640, 480, true, true>',
    'S2/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, false, true> + warp_sparse_depth_kernel',
    'S2/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 1, true>',
    'S2/forward/C2': '2: frame_params_tiles_kernel + warp_forward_kernel<2, false, false>',
    'S2/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 3, true>',
    'S2/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<640, 480, 1, true>',
    'S2/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 3, true>',
    'S2/forward/C3/bicubic': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    'S2/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, true, false, true>',
    'S2/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, false, false, true>',
    'S2/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, true, true, false>',
    'S2/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, false, true, false>',
    'S2/unwarp_normals/params': '1: unwarp_normals_shear_kernel<640, 480, true, false, true>',
    'S2/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, false, false, true>',
    'S2/channels_last/forward': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<640, 480, false>',
    'S2/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<640, 480, true>',
    'S2/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<640, 480, true>',
    'S2/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<640, 480, false>',
    'S2/warp_normal_image': '2: frame_params_kernel + warp_forward_kernel<3, false, true>',
    'S2/warp_with_homography': '2: frame_params_from_h_kernel + warp_forward_kernel<3, false, false>',
    'S2/warp_rgbd_packed': '2: frame_params_kernel + warp_rgbd_nhwc4_kernel',
    'S2/smaller_input/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_fast_kernel<0, 0, true>',
    'S2/smaller_input/forward/C3': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    'S2/strided/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_fast_kernel<0, 0, true>',
    'S2/strided/forward/C3': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    'S2/strided/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
    'S2/offset_in/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
    'S2/offset_in/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 3, true>',
    'S2/offset_in/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, true, false, true>',
    'S2/offset_in/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, false, true> + warp_sparse_depth_kernel',
    'S2/offset_out/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_fast_kernel<640, 480, true>',
    'S2/offset_out/forward/C3': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    'S2/offset_out/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
    'S2/offset_out/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + memset + warp_rgbd_fast_kernel<640, 480, false> + warp_sparse_depth_kernel',
    'S1/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, true, true>',
    'S1/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, false, true>',
    'S1/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, true, true>',
    'S1/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, true, true>',
    'S1/prepare': '1: frame_params_tiles_kernel',
    'S1/warp_rgbd/params': '1: warp_rgbd_shear_kernel<320, 240, true, true>',
    'S1/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, false, true> + warp_sparse_depth_kernel',
    'S1/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<320, 240, 1, true>',
    'S1/forward/C2': '2: frame_params_tiles_kernel + warp_forward_kernel<2, false, false>',
    'S1/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<320, 240, 3, true>',
    'S1/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<320, 240, 1, true>',
    'S1/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<320, 240, 3, true>',
    'S1/forward/C3/bicubic': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    'S1/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, true, false, true>',
    'S1/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, false, false, true>',
    'S1/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, true, true, false>',
    'S1/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, false, true, false>',
    'S1/unwarp_normals/params': '1: unwarp_normals_shear_kernel<320, 240, true, false, true>',
    'S1/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, false, false, true>',
    'S1/channels_last/forward': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<320, 240, false>',
    'S1/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<320, 240, true>',
    'S1/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<320, 240, true>',
    'S1/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<320, 240, false>',
    '640x489/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, true, true>',
    '640x489/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, false, true>',
    '640x489/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, true, true>',
    '640x489/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, true, true>',
    '640x489/prepare': '1: frame_params_tiles_kernel',
    '640x489/warp_rgbd/params': '1: warp_rgbd_shear_kernel<640, 489, true, true>',
    '640x489/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, false, true> + warp_sparse_depth_kernel',
    '640x489/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 489, 1, true>',
    '640x489/forward/C2': '2: frame_params_tiles_kernel + warp_forward_kernel<2, false, false>',
    '640x489/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 489, 3, true>',
    '640x489/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<640, 489, 1, true>',
    '640x489/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 489, 3, true>',
    '640x489/forward/C3/bicubic': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    '640x489/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, true, false, true>',
    '640x489/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, false, false, true>',
    '640x489/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, true, true, false>',
    '640x489/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, false, true, false>',
    '640x489/unwarp_normals/params': '1: unwarp_normals_shear_kernel<640, 489, true, false, true>',
    '640x489/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, false, false, true>',
    '640x489/channels_last/forward': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<0, 0, false>',
    '640x489/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<0, 0, true>',
    '640x489/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<0, 0, true>',
    '640x489/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<0, 0, false>',
    '416x301/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, true, true>',
    '416x301/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, false, true>',
    '416x301/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, true, true>',
    '416x301/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, true, true>',
    '416x301/prepare': '1: frame_params_tiles_kernel',
    '416x301/warp_rgbd/params': '1: warp_rgbd_shear_kernel<0, 0, true, true>',
    '416x301/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, false, true> + warp_sparse_depth_kernel',
    '416x301/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<0, 0, 1, true>',
    '416x301/forward/C2': '2: frame_params_tiles_kernel + warp_forward_kernel<2, false, false>',
    '416x301/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<0, 0, 3, true>',
    '416x301/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<0, 0, 1, true>',
    '416x301/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<0, 0, 3, true>',
    '416x301/forward/C3/bicubic': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    '416x301/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, true, false, true>',
    '416x301/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, false, false, true>',
    '416x301/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, true, true, false>',
    '416x301/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, false, true, false>',
    '416x301/unwarp_normals/params': '1: unwarp_normals_shear_kernel<0, 0, true, false, true>',
    '416x301/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, false, false, true>',
    '416x301/channels_last/forward': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<0, 0, false>',
    '416x301/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_cl_kernel<0, 0, true>',
    '416x301/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<0, 0, true>',
    '416x301/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_cl_kernel<0, 0, false>',
    '300x201/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_fast_kernel<0, 0, true>',
    '300x201/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_fast_kernel<0, 0, false>',
    '300x201/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_fast_kernel<0, 0, true>',
    '300x201/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_fast_kernel<0, 0, true>',
    '300x201/prepare': '1: frame_params_tiles_kernel',
    '300x201/warp_rgbd/params': '1: warp_rgbd_fast_kernel<0, 0, true>',
    '300x201/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + memset + warp_rgbd_fast_kernel<0, 0, false> + warp_sparse_depth_kernel',
    '300x201/forward/C1': '2: frame_params_tiles_kernel + warp_forward_kernel<1, false, false>',
    '300x201/forward/C2': '2: frame_params_tiles_kernel + warp_forward_kernel<2, false, false>',
    '300x201/forward/C3': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    '300x201/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
    '300x201/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    '300x201/forward/C3/bicubic': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    '300x201/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
    '300x201/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
    '300x201/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
    '300x201/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
    '300x201/unwarp_normals/params': '1: unwarp_normals_fast_kernel<0, 0, true>',
    '300x201/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
    '300x201/channels_last/forward': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
    '300x201/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_forward_kernel<3, true, false>',
    '300x201/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
    '300x201/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
}
DIFFERS = {
    'shear0': {
        'S2/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<640, 480, true>',
        'S2/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_fast_kernel<640, 480, false>',
        'S2/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_fast_kernel<640, 480, true>',
        'S2/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_fast_kernel<640, 480, true>',
        'S2/prepare': '1: frame_params_kernel',
        'S2/warp_rgbd/params': '1: warp_rgbd_fast_kernel<640, 480, true>',
        'S2/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<640, 480, false> + warp_sparse_depth_kernel',
        'S2/forward/C1': '2: frame_params_kernel + warp_forward_kernel<1, false, false>',
        'S2/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        'S2/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
        'S2/forward/C3/nearest': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
        'S2/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, false>',
        'S2/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
        'S2/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, false>',
        'S2/unwarp_normals/params': '1: unwarp_normals_fast_kernel<640, 480, true>',
        'S2/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, false>',
        'S2/channels_last/forward': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/channels_last/warp_rgbd': '2: frame_params_kernel + warp_forward_kernel<3, true, false>',
        'S2/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        'S2/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        'S2/smaller_input/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        'S2/smaller_input/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/strided/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        'S2/strided/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/offset_in/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<640, 480, true>',
        'S2/offset_in/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/offset_in/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
        'S2/offset_in/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<640, 480, false> + warp_sparse_depth_kernel',
        'S2/offset_out/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<640, 480, true>',
        'S2/offset_out/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/offset_out/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<640, 480, false> + warp_sparse_depth_kernel',
        'S1/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<320, 240, true>',
        'S1/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_fast_kernel<320, 240, false>',
        'S1/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_fast_kernel<320, 240, true>',
        'S1/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_fast_kernel<320, 240, true>',
        'S1/prepare': '1: frame_params_kernel',
        'S1/warp_rgbd/params': '1: warp_rgbd_fast_kernel<320, 240, true>',
        'S1/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<320, 240, false> + warp_sparse_depth_kernel',
        'S1/forward/C1': '2: frame_params_kernel + warp_forward_kernel<1, false, false>',
        'S1/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        'S1/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S1/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
        'S1/forward/C3/nearest': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S1/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S1/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, true>',
        'S1/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, false>',
        'S1/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, true>',
        'S1/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, false>',
        'S1/unwarp_normals/params': '1: unwarp_normals_fast_kernel<320, 240, true>',
        'S1/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, false>',
        'S1/channels_last/forward': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S1/channels_last/warp_rgbd': '2: frame_params_kernel + warp_forward_kernel<3, true, false>',
        'S1/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        'S1/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '640x489/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '640x489/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, false>',
        '640x489/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '640x489/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '640x489/prepare': '1: frame_params_kernel',
        '640x489/warp_rgbd/params': '1: warp_rgbd_fast_kernel<0, 0, true>',
        '640x489/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<0, 0, false> + warp_sparse_depth_kernel',
        '640x489/forward/C1': '2: frame_params_kernel + warp_forward_kernel<1, false, false>',
        '640x489/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        '640x489/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '640x489/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
        '640x489/forward/C3/nearest': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '640x489/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '640x489/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '640x489/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '640x489/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '640x489/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '640x489/unwarp_normals/params': '1: unwarp_normals_fast_kernel<0, 0, true>',
        '640x489/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '640x489/channels_last/forward': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '640x489/channels_last/warp_rgbd': '2: frame_params_kernel + warp_forward_kernel<3, true, false>',
        '640x489/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        '640x489/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '416x301/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '416x301/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, false>',
        '416x301/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '416x301/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '416x301/prepare': '1: frame_params_kernel',
        '416x301/warp_rgbd/params': '1: warp_rgbd_fast_kernel<0, 0, true>',
        '416x301/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<0, 0, false> + warp_sparse_depth_kernel',
        '416x301/forward/C1': '2: frame_params_kernel + warp_forward_kernel<1, false, false>',
        '416x301/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        '416x301/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '416x301/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
        '416x301/forward/C3/nearest': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '416x301/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '416x301/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '416x301/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '416x301/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '416x301/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '416x301/unwarp_normals/params': '1: unwarp_normals_fast_kernel<0, 0, true>',
        '416x301/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '416x301/channels_last/forward': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '416x301/channels_last/warp_rgbd': '2: frame_params_kernel + warp_forward_kernel<3, true, false>',
        '416x301/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        '416x301/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '300x201/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '300x201/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, false>',
        '300x201/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '300x201/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '300x201/prepare': '1: frame_params_kernel',
        '300x201/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<0, 0, false> + warp_sparse_depth_kernel',
        '300x201/forward/C1': '2: frame_params_kernel + warp_forward_kernel<1, false, false>',
        '300x201/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        '300x201/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
        '300x201/forward/C3/nearest': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/channels_last/forward': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/channels_last/warp_rgbd': '2: frame_params_kernel + warp_forward_kernel<3, true, false>',
    },
    'shear1': {
        'S2/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
        'S2/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, false>',
        'S2/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
        'S2/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, false>',
        'S2/unwarp_normals/params': '1: unwarp_normals_fast_kernel<640, 480, true>',
        'S2/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, false>',
        'S2/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        'S2/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        'S2/offset_in/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<640, 480, true>',
        'S1/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, true>',
        'S1/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, false>',
        'S1/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, true>',
        'S1/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, false>',
        'S1/unwarp_normals/params': '1: unwarp_normals_fast_kernel<320, 240, true>',
        'S1/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<320, 240, false>',
        'S1/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        'S1/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '640x489/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '640x489/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '640x489/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '640x489/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '640x489/unwarp_normals/params': '1: unwarp_normals_fast_kernel<0, 0, true>',
        '640x489/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '640x489/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        '640x489/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '416x301/unwarp_normals': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '416x301/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '416x301/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, true>',
        '416x301/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '416x301/unwarp_normals/params': '1: unwarp_normals_fast_kernel<0, 0, true>',
        '416x301/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_fast_kernel<0, 0, false>',
        '416x301/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        '416x301/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
    },
    'tma': {
        'S2/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S2/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false>',
        'S2/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S2/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S2/warp_rgbd/params': '1: warp_rgbd_tma_kernel<true>',
        'S2/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false> + warp_sparse_depth_kernel',
        'S2/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        'S2/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        'S2/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        'S2/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        'S2/unwarp_normals/params': '1: unwarp_normals_tma_kernel<true>',
        'S2/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        'S2/smaller_input/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S2/strided/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S2/strided/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        'S2/offset_in/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + memset + warp_rgbd_shear_kernel<640, 480, false, true> + warp_sparse_depth_kernel',
        'S2/offset_out/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S2/offset_out/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        'S2/offset_out/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false> + warp_sparse_depth_kernel',
        'S1/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S1/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false>',
        'S1/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S1/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        'S1/warp_rgbd/params': '1: warp_rgbd_tma_kernel<true>',
        'S1/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false> + warp_sparse_depth_kernel',
        'S1/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        'S1/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        'S1/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        'S1/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        'S1/unwarp_normals/params': '1: unwarp_normals_tma_kernel<true>',
        'S1/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '640x489/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '640x489/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false>',
        '640x489/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '640x489/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '640x489/warp_rgbd/params': '1: warp_rgbd_tma_kernel<true>',
        '640x489/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false> + warp_sparse_depth_kernel',
        '640x489/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        '640x489/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '640x489/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        '640x489/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '640x489/unwarp_normals/params': '1: unwarp_normals_tma_kernel<true>',
        '640x489/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '416x301/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '416x301/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false>',
        '416x301/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '416x301/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '416x301/warp_rgbd/params': '1: warp_rgbd_tma_kernel<true>',
        '416x301/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false> + warp_sparse_depth_kernel',
        '416x301/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        '416x301/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '416x301/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        '416x301/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '416x301/unwarp_normals/params': '1: unwarp_normals_tma_kernel<true>',
        '416x301/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '300x201/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '300x201/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false>',
        '300x201/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '300x201/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_tma_kernel<true>',
        '300x201/warp_rgbd/params': '1: warp_rgbd_tma_kernel<true>',
        '300x201/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_tma_kernel<false> + warp_sparse_depth_kernel',
        '300x201/unwarp_normals': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        '300x201/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '300x201/unwarp_normals/valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<true>',
        '300x201/unwarp_normals/raw_valid': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
        '300x201/unwarp_normals/params': '1: unwarp_normals_tma_kernel<true>',
        '300x201/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_tma_kernel<false>',
    },
    'inv_box': {
        'S2/unwarp_normals': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<640, 480, true, false>',
        'S2/unwarp_normals/raw': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<640, 480, false, false>',
        'S2/unwarp_normals/valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<640, 480, true, true>',
        'S2/unwarp_normals/raw_valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<640, 480, false, true>',
        'S2/inverse_warp_normal_image': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<640, 480, false, false>',
        'S2/offset_out/unwarp_normals': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<640, 480, true, false>',
        'S1/unwarp_normals': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<320, 240, true, false>',
        'S1/unwarp_normals/raw': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<320, 240, false, false>',
        'S1/unwarp_normals/valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<320, 240, true, true>',
        'S1/unwarp_normals/raw_valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<320, 240, false, true>',
        'S1/inverse_warp_normal_image': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<320, 240, false, false>',
        '640x489/unwarp_normals': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, true, false>',
        '640x489/unwarp_normals/raw': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, false>',
        '640x489/unwarp_normals/valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, true, true>',
        '640x489/unwarp_normals/raw_valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, true>',
        '640x489/inverse_warp_normal_image': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, false>',
        '416x301/unwarp_normals': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, true, false>',
        '416x301/unwarp_normals/raw': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, false>',
        '416x301/unwarp_normals/valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, true, true>',
        '416x301/unwarp_normals/raw_valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, true>',
        '416x301/inverse_warp_normal_image': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, false>',
        '300x201/unwarp_normals': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, true, false>',
        '300x201/unwarp_normals/raw': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, false>',
        '300x201/unwarp_normals/valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, true, true>',
        '300x201/unwarp_normals/raw_valid': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, true>',
        '300x201/inverse_warp_normal_image': '2: frame_params_inv_boxes_kernel + unwarp_normals_box_kernel<0, 0, false, false>',
    },
    'tma_store0': {
        'S2/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, false>',
        'S2/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, false, false>',
        'S2/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, false>',
        'S2/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, false>',
        'S2/warp_rgbd/params': '1: warp_rgbd_shear_kernel<640, 480, true, false>',
        'S2/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, false, false> + warp_sparse_depth_kernel',
        'S2/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 1, false>',
        'S2/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 3, false>',
        'S2/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<640, 480, 1, false>',
        'S2/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 3, false>',
        'S2/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, true, false, false>',
        'S2/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, false, false, false>',
        'S2/unwarp_normals/params': '1: unwarp_normals_shear_kernel<640, 480, true, false, false>',
        'S2/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, false, false, false>',
        'S2/channels_last/forward': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
        'S2/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_forward_kernel<3, true, false>',
        'S2/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        'S2/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        'S2/offset_in/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, true, false>',
        'S2/offset_in/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 480, 3, false>',
        'S2/offset_in/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 480, true, false, false>',
        'S2/offset_in/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 480, false, false> + warp_sparse_depth_kernel',
        'S1/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, true, false>',
        'S1/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, false, false>',
        'S1/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, true, false>',
        'S1/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, true, false>',
        'S1/warp_rgbd/params': '1: warp_rgbd_shear_kernel<320, 240, true, false>',
        'S1/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<320, 240, false, false> + warp_sparse_depth_kernel',
        'S1/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<320, 240, 1, false>',
        'S1/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<320, 240, 3, false>',
        'S1/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<320, 240, 1, false>',
        'S1/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<320, 240, 3, false>',
        'S1/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, true, false, false>',
        'S1/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, false, false, false>',
        'S1/unwarp_normals/params': '1: unwarp_normals_shear_kernel<320, 240, true, false, false>',
        'S1/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<320, 240, false, false, false>',
        'S1/channels_last/forward': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
        'S1/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_forward_kernel<3, true, false>',
        'S1/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        'S1/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '640x489/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, true, false>',
        '640x489/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, false, false>',
        '640x489/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, true, false>',
        '640x489/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, true, false>',
        '640x489/warp_rgbd/params': '1: warp_rgbd_shear_kernel<640, 489, true, false>',
        '640x489/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<640, 489, false, false> + warp_sparse_depth_kernel',
        '640x489/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 489, 1, false>',
        '640x489/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 489, 3, false>',
        '640x489/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<640, 489, 1, false>',
        '640x489/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<640, 489, 3, false>',
        '640x489/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, true, false, false>',
        '640x489/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, false, false, false>',
        '640x489/unwarp_normals/params': '1: unwarp_normals_shear_kernel<640, 489, true, false, false>',
        '640x489/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<640, 489, false, false, false>',
        '640x489/channels_last/forward': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
        '640x489/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_forward_kernel<3, true, false>',
        '640x489/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        '640x489/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
        '416x301/warp_rgbd': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, true, false>',
        '416x301/warp_rgbd/no_depth': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, false, false>',
        '416x301/warp_rgbd/coverage': '2: memset + frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, true, false>',
        '416x301/warp_rgbd/nearest': '2: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, true, false>',
        '416x301/warp_rgbd/params': '1: warp_rgbd_shear_kernel<0, 0, true, false>',
        '416x301/warp_rgb_sparse_depth': '3: frame_params_tiles_kernel + warp_rgbd_shear_kernel<0, 0, false, false> + warp_sparse_depth_kernel',
        '416x301/forward/C1': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<0, 0, 1, false>',
        '416x301/forward/C3': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<0, 0, 3, false>',
        '416x301/forward/C5': '3: frame_params_tiles_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<0, 0, 1, false>',
        '416x301/forward/C3/nearest': '2: frame_params_tiles_kernel + warp_planes_shear_kernel<0, 0, 3, false>',
        '416x301/unwarp_normals': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, true, false, false>',
        '416x301/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, false, false, false>',
        '416x301/unwarp_normals/params': '1: unwarp_normals_shear_kernel<0, 0, true, false, false>',
        '416x301/inverse_warp_normal_image': '2: frame_params_kernel + unwarp_normals_shear_kernel<0, 0, false, false, false>',
        '416x301/channels_last/forward': '2: frame_params_tiles_kernel + warp_forward_kernel<3, false, false>',
        '416x301/channels_last/warp_rgbd': '2: frame_params_tiles_kernel + warp_forward_kernel<3, true, false>',
        '416x301/channels_last/unwarp_normals': '2: frame_params_kernel + unwarp_normals_kernel<true>',
        '416x301/channels_last/unwarp_normals/raw': '2: frame_params_kernel + unwarp_normals_kernel<false>',
    },
    'tile_skip0': {
        'S2/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
        'S2/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 480, false, true>',
        'S2/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
        'S2/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
        'S2/prepare': '1: frame_params_kernel',
        'S2/warp_rgb_sparse_depth': '3: frame_params_kernel + warp_rgbd_shear_kernel<640, 480, false, true> + warp_sparse_depth_kernel',
        'S2/forward/C1': '2: frame_params_kernel + warp_planes_shear_kernel<640, 480, 1, true>',
        'S2/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        'S2/forward/C3': '2: frame_params_kernel + warp_planes_shear_kernel<640, 480, 3, true>',
        'S2/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<640, 480, 1, true>',
        'S2/forward/C3/nearest': '2: frame_params_kernel + warp_planes_shear_kernel<640, 480, 3, true>',
        'S2/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/channels_last/forward': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<640, 480, false>',
        'S2/channels_last/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<640, 480, true>',
        'S2/smaller_input/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        'S2/smaller_input/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/strided/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        'S2/strided/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/offset_in/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 480, true, true>',
        'S2/offset_in/forward/C3': '2: frame_params_kernel + warp_planes_shear_kernel<640, 480, 3, true>',
        'S2/offset_in/warp_rgb_sparse_depth': '3: frame_params_kernel + warp_rgbd_shear_kernel<640, 480, false, true> + warp_sparse_depth_kernel',
        'S2/offset_out/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<640, 480, true>',
        'S2/offset_out/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S2/offset_out/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<640, 480, false> + warp_sparse_depth_kernel',
        'S1/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_kernel<320, 240, true, true>',
        'S1/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_shear_kernel<320, 240, false, true>',
        'S1/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_kernel<320, 240, true, true>',
        'S1/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_shear_kernel<320, 240, true, true>',
        'S1/prepare': '1: frame_params_kernel',
        'S1/warp_rgb_sparse_depth': '3: frame_params_kernel + warp_rgbd_shear_kernel<320, 240, false, true> + warp_sparse_depth_kernel',
        'S1/forward/C1': '2: frame_params_kernel + warp_planes_shear_kernel<320, 240, 1, true>',
        'S1/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        'S1/forward/C3': '2: frame_params_kernel + warp_planes_shear_kernel<320, 240, 3, true>',
        'S1/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<320, 240, 1, true>',
        'S1/forward/C3/nearest': '2: frame_params_kernel + warp_planes_shear_kernel<320, 240, 3, true>',
        'S1/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        'S1/channels_last/forward': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<320, 240, false>',
        'S1/channels_last/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<320, 240, true>',
        '640x489/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 489, true, true>',
        '640x489/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 489, false, true>',
        '640x489/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_kernel<640, 489, true, true>',
        '640x489/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_shear_kernel<640, 489, true, true>',
        '640x489/prepare': '1: frame_params_kernel',
        '640x489/warp_rgb_sparse_depth': '3: frame_params_kernel + warp_rgbd_shear_kernel<640, 489, false, true> + warp_sparse_depth_kernel',
        '640x489/forward/C1': '2: frame_params_kernel + warp_planes_shear_kernel<640, 489, 1, true>',
        '640x489/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        '640x489/forward/C3': '2: frame_params_kernel + warp_planes_shear_kernel<640, 489, 3, true>',
        '640x489/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<640, 489, 1, true>',
        '640x489/forward/C3/nearest': '2: frame_params_kernel + warp_planes_shear_kernel<640, 489, 3, true>',
        '640x489/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '640x489/channels_last/forward': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<0, 0, false>',
        '640x489/channels_last/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<0, 0, true>',
        '416x301/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_kernel<0, 0, true, true>',
        '416x301/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_shear_kernel<0, 0, false, true>',
        '416x301/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_shear_kernel<0, 0, true, true>',
        '416x301/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_shear_kernel<0, 0, true, true>',
        '416x301/prepare': '1: frame_params_kernel',
        '416x301/warp_rgb_sparse_depth': '3: frame_params_kernel + warp_rgbd_shear_kernel<0, 0, false, true> + warp_sparse_depth_kernel',
        '416x301/forward/C1': '2: frame_params_kernel + warp_planes_shear_kernel<0, 0, 1, true>',
        '416x301/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        '416x301/forward/C3': '2: frame_params_kernel + warp_planes_shear_kernel<0, 0, 3, true>',
        '416x301/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_planes_shear_kernel<0, 0, 1, true>',
        '416x301/forward/C3/nearest': '2: frame_params_kernel + warp_planes_shear_kernel<0, 0, 3, true>',
        '416x301/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '416x301/channels_last/forward': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<0, 0, false>',
        '416x301/channels_last/warp_rgbd': '2: frame_params_kernel + warp_rgbd_shear_cl_kernel<0, 0, true>',
        '300x201/warp_rgbd': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '300x201/warp_rgbd/no_depth': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, false>',
        '300x201/warp_rgbd/coverage': '2: memset + frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '300x201/warp_rgbd/nearest': '2: frame_params_kernel + warp_rgbd_fast_kernel<0, 0, true>',
        '300x201/prepare': '1: frame_params_kernel',
        '300x201/warp_rgb_sparse_depth': '3: frame_params_kernel + memset + warp_rgbd_fast_kernel<0, 0, false> + warp_sparse_depth_kernel',
        '300x201/forward/C1': '2: frame_params_kernel + warp_forward_kernel<1, false, false>',
        '300x201/forward/C2': '2: frame_params_kernel + warp_forward_kernel<2, false, false>',
        '300x201/forward/C3': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/forward/C5': '3: frame_params_kernel + warp_forward_kernel<4, false, false> + warp_forward_kernel<1, false, false>',
        '300x201/forward/C3/nearest': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/forward/C3/bicubic': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/channels_last/forward': '2: frame_params_kernel + warp_forward_kernel<3, false, false>',
        '300x201/channels_last/warp_rgbd': '2: frame_params_kernel + warp_forward_kernel<3, true, false>',
    },
}


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    if "--child" in sys.argv:
        _child()
    elif "--freeze" in sys.argv:
        _freeze()
