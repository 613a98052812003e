"""The validity plane of the inverse warp, unwarp_normals(..., with_valid=True), bit for bit.

valid[b, Y, X] is 1 exactly when one of the four bilinear taps of camera pixel (X, Y) -- x0 or x0 + 1 by y0 or y0 + 1, with
(x0, y0) = floor of its canvas coordinate, a non-finite coordinate reading as -100 -- lies inside the canvas, whatever the
tap's weight (tests/exact_reference.py: touch_plane).  Where valid is 0 and the frame's R is finite, z is +0 in all three
channels.  Six kernel families write the plane; each case records with torch.profiler which one ran and the test holds it to
the family it is meant to reach.  The kernel switches are read once per process, so each setting runs its cases in a fresh
process with VIDC_* stripped from the inherited environment."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SETTINGS = {"default": {}, "shear0": {"VIDC_SHEAR": "0"}, "shear1": {"VIDC_SHEAR": "1"}, "tma": {"VIDC_TMA": "1"},
            "inv_box": {"VIDC_INV_BOX": "1"}, "tma_store0": {"VIDC_TMA_STORE": "0"}}
CANVASES = {"S2": (404.0, 404.0, 319.87654, 239.87603), "S1": (202.0, 202.0, 159.93827, 119.938015),
            "640x489": (404.0, 404.0, 319.87654, 244.4), "416x301": (300.0, 300.0, 207.7, 150.2),
            "300x201": (250.0, 250.0, 149.7, 100.2), "tiny": (40.4, 40.4, 31.9, 23.9)}

# the unwarp kernel each case must reach (prefix of its demangled name), per setting
_SHEAR = {"S2": "unwarp_normals_shear_kernel<640, 480, ", "S1": "unwarp_normals_shear_kernel<320, 240, ",
          "640x489": "unwarp_normals_shear_kernel<640, 489, ", "416x301": "unwarp_normals_shear_kernel<0, 0, ",
          "300x201": "unwarp_normals_fast_kernel<0, 0, ", "tiny": "unwarp_normals_shear_kernel<"}
DEFAULT = dict({f"{c}/{n}": k for c, k in _SHEAR.items() for n in ("norm", "raw")},
               **{"S2/params": _SHEAR["S2"], "S1/special": _SHEAR["S1"], "tiny/degenerate": _SHEAR["tiny"],
                  "tiny/exact_edges": _SHEAR["tiny"], "S1/isolated": _SHEAR["S1"], "S2/channels_last": "unwarp_normals_kernel<",
                  "S2/column_stride": "unwarp_normals_kernel<", "S2/padded_rows": "unwarp_normals_fast_kernel<0, 0, ",
                  "S2/valid_offset0": _SHEAR["S2"], "S2/valid_offset1": "unwarp_normals_fast_kernel<640, 480, ",
                  "S2/valid_offset2": "unwarp_normals_fast_kernel<640, 480, ", "S2/valid_offset3": "unwarp_normals_fast_kernel<640, 480, "})
# the other settings run the canvas cases only
_CANVAS_CASES = [f"{c}/{n}" for c in ("S2", "S1", "640x489", "300x201") for n in ("norm", "raw")] + ["S1/special"]
EXPECTED = {
    "default": DEFAULT,
    "shear0": {k: "unwarp_normals_fast_kernel<" for k in _CANVAS_CASES},
    "shear1": {k: "unwarp_normals_fast_kernel<" for k in _CANVAS_CASES},
    "tma": {k: "unwarp_normals_tma_kernel<" for k in _CANVAS_CASES},
    "inv_box": {k: "unwarp_normals_box_kernel<" for k in _CANVAS_CASES},
    "tma_store0": {k: DEFAULT[k] for k in _CANVAS_CASES},
}


def _child(setting):
    import ctypes

    import numpy as np
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    from oracle import oracle as O
    from tests import common as C
    from tests import exact_reference as X
    from tests.test_exact_reference import exact_edge_gravity
    from vi_depth_completion_b200._cabi import check, lib
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment, _image, _stream_ptr

    dev = torch.device("cuda", 0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    wanted = EXPECTED[setting]
    seen = {}

    def record(name, fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        seen[name] = [e.name.split("(")[0].removeprefix("void ").removeprefix("vidc_k::").strip()
                      for e in prof.events() if e.device_type == DeviceType.CUDA and "unwarp_normals" in e.name]
        return out

    def check_plane(name, o, I_g, I_a, valid, z):
        want = X.touch_plane(o, I_g, I_a)
        got = valid.cpu().numpy().reshape(want.shape)
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"{setting} {name}: {len(bad)} validity flags differ from the touch plane, first {tuple(bad[0])}"
        _, R, _ = o.build_homography(I_g, I_a)
        zn = z.cpu().numpy()
        for b in range(want.shape[0]):
            if np.isfinite(R[b]).all():
                zb = C.bits(zn[b])[:, want[b] == 0]
                assert (zb == 0).all(), f"{setting} {name}: frame {b}: z is not +0 where valid is 0"
        return int((want == 0).sum())

    def steep(seed):
        """two moderate frames, two near +-90 deg roll (column-major / along-Y tiles), two steep-pitch frames whose camera
        images partly map outside the canvas (valid 0 there)"""
        g_r, a_r = C.random_gravity(2, seed=seed, roll_deg=30, pitch_deg=30)
        g_x, a_x = C.extreme_roll_gravity(7, 3)
        g_i, a_i = C.isolated_nonfinite_gravity()
        return np.concatenate([g_r, g_x[[3, 5]], g_i[:2]]), np.concatenate([a_r, a_x[[3, 5]], a_i[:2]])

    zeros = 0
    for canvas, intr in CANVASES.items():
        cases = [k for k in wanted if k.startswith(canvas + "/")]
        if not cases:
            continue
        w, o = Warping2DOFAlignment(*intr), O.Oracle(*intr)
        I_g, I_a = steep(len(seen) + 3)
        B = I_g.shape[0]
        nrm = C.random_images(B, o.H, o.W, 6)[2]
        for name in cases:
            kind = name.split("/", 1)[1]
            g, a = I_g, I_a
            if kind in ("norm", "raw"):
                _, z, valid = record(name, lambda: w.unwarp_normals(t(nrm), t(g), t(a), normalize=kind == "norm", with_valid=True))
                zeros += check_plane(name, o, g, a, valid, z if kind == "raw" else w.unwarp_normals(t(nrm), t(g), t(a), normalize=False)[1])
            elif kind == "params":
                p = w.prepare(t(g), t(a))
                _, z, valid = record(name, lambda: w.unwarp_normals(t(nrm), params=p, normalize=False, with_valid=True))
                zeros += check_plane(name, o, g, a, valid, z)
            elif kind == "special":
                img = C.special_value_images(4, o.H, o.W, 21)[2]
                g, a = C.special_value_gravity(4)
                _, z, valid = record(name, lambda: w.unwarp_normals(t(img), t(g), t(a), normalize=False, with_valid=True))
                zeros += check_plane(name, o, g, a, valid, z)
            elif kind in ("degenerate", "exact_edges", "isolated"):
                g, a = {"degenerate": C.degenerate_gravity, "exact_edges": exact_edge_gravity, "isolated": C.isolated_nonfinite_gravity}[kind]()
                img = C.random_images(g.shape[0], o.H, o.W, 7)[2]
                _, z, valid = record(name, lambda: w.unwarp_normals(t(img), t(g), t(a), normalize=False, with_valid=True))
                zeros += check_plane(name, o, g, a, valid, z)
            elif kind in ("channels_last", "column_stride", "padded_rows"):
                x = t(nrm)
                if kind == "channels_last":
                    x = x.contiguous(memory_format=torch.channels_last)
                elif kind == "column_stride":
                    wide = torch.zeros(B, 3, o.H, 2 * o.W, device=dev); wide[..., ::2] = x; x = wide[..., ::2]
                else:
                    wide = torch.zeros(B, 3, o.H, o.W + 64, device=dev); wide[..., :o.W] = x; x = wide[..., :o.W]
                _, z, valid = record(name, lambda: w.unwarp_normals(x, t(g), t(a), normalize=False, with_valid=True))
                zeros += check_plane(name, o, g, a, valid, z)
            elif kind.startswith("valid_offset"):
                # the plane 0..3 bytes past a 4-byte boundary of a guarded buffer: the sheared kernel stores it two bytes at a
                # time and takes only a 4-byte aligned plane; nothing may be written outside it
                off, guard, n = int(kind[-1]), 256, B * o.H * o.W
                buf = torch.full((n + 2 * guard + 4,), 0xA5, dtype=torch.uint8, device=dev)
                z = torch.empty(B, 3, o.H, o.W, device=dev)
                gd, ad, x = t(g), t(a), t(nrm)
                ws, Hout = w._params_ws(B, dev), torch.empty(B, 3, 3, device=dev)
                record(name, lambda: check(lib().vidc_unwarp_normals(ctypes.byref(w._cam), ctypes.byref(_image(x)), gd.data_ptr(),
                                                                     ad.data_ptr(), B, 0, ws.data_ptr(), Hout.data_ptr(),
                                                                     ctypes.byref(_image(z)), buf.data_ptr() + guard + off,
                                                                     _stream_ptr(dev))))
                host = buf.cpu().numpy()
                assert (host[:guard + off] == 0xA5).all() and (host[guard + off + n:] == 0xA5).all(), f"{name}: write outside the plane"
                zeros += check_plane(name, o, g, a, torch.from_numpy(host[guard + off:guard + off + n].copy()), z)
    assert zeros > 0, "no case has an untouched pixel"
    print(json.dumps(seen), flush=True)


def _run(setting):
    env = {k: v for k, v in os.environ.items() if not k.startswith("VIDC_")}
    env.update(SETTINGS[setting])
    res = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", setting], cwd=ROOT, env=env, capture_output=True,
                         text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    return json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])


@pytest.mark.gpu
@pytest.mark.parametrize("setting", list(SETTINGS))
def test_validity_plane_is_the_touch_plane(cuda_device, setting):
    seen, want = _run(setting), EXPECTED[setting]
    assert set(seen) == set(want)
    bad = [f"{k}: want one {want[k]}..., ran {seen[k]}" for k in sorted(want) if len(seen[k]) != 1 or not seen[k][0].startswith(want[k])]
    assert not bad, f"{setting}: cases reached other kernels:\n" + "\n".join(bad)
    print(f"[validity] {setting}: " + "; ".join(f"{k} -> {seen[k][0]}" for k in sorted(seen)))


if __name__ == "__main__" and sys.argv[1:2] == ["--child"]:
    sys.path.insert(0, ROOT)
    _child(sys.argv[2])
