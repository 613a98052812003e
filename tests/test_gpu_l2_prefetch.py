"""The L2 prefetch of the sheared kernels is a hint: no output bit may depend on it.

The prefetch switches (VIDC_PF_BULK, VIDC_INV_PF_WAVES_X100, VIDC_FWD_PF_WAVES_X100) are read once per process, so every
variant runs the same workloads in a fresh process and prints a SHA-256 of every output: the forward warp's RGB, depth, mask
and coverage, the inverse warp's normals, and the reference-shaped RGB warp.  Inputs offset by one float (no tensor map can
describe them, so the bulk prefetch is not used) must give the same bits as aligned ones."""
import hashlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (name, camera, gravity): S2 (the bench workload), S3 at rolls up to +-90 deg (lanes along Y), S1 (320x240), the 640x489
# compile-time canvas and a runtime-geometry canvas (416x301)
WORKLOADS = [("S2", "S2", ("random", 24, 1234, 30, 30)), ("S3", "S3", ("roll", 24, 5)), ("S1", "S1", ("random", 8, 1234, 30, 30)),
             ("640x489", (404.0, 404.0, 319.87654, 244.4), ("random", 8, 33, 60, 20)),
             ("416x301", (300.0, 300.0, 207.7, 150.2), ("random", 8, 7, 45, 30))]


def _digest(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def _child():
    import torch
    from tests import common as C
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    dev = torch.device("cuda", 0)
    out = {}
    for name, cam, grav in WORKLOADS:
        w = Warping2DOFAlignment(*(C.CAMERAS[cam] if isinstance(cam, str) else cam))
        H, W = int(w.H), int(w.W)
        if grav[0] == "roll":
            I_g, I_a = C.extreme_roll_gravity(grav[1], seed=grav[2])
        else:
            I_g, I_a = C.random_gravity(grav[1], seed=grav[2], roll_deg=grav[3], pitch_deg=grav[4])
        B = I_g.shape[0]
        g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)
        gen = torch.Generator(device=dev).manual_seed(11)
        rgb = torch.rand(B, 3, H, W, device=dev, generator=gen)
        depth = torch.rand(B, 1, H, W, device=dev, generator=gen) * 9.6 + 0.4
        nrm = torch.randn(B, 3, H, W, device=dev, generator=gen)

        def offset(t):                                   # same values, data pointer one float past a 16-byte boundary
            buf = torch.empty(t.numel() + 4, device=dev)
            v = buf[1:1 + t.numel()].view(t.shape)
            v.copy_(t)
            return v

        for tag, (x_rgb, x_dep, x_nrm) in (("", (rgb, depth, nrm)), ("+1", (offset(rgb), offset(depth), offset(nrm)))):
            p = w.prepare(g, a)
            _, rgb_w, dep_w, mask = w.warp_rgbd(x_rgb, x_dep, params=p)
            _, n_hat = w.unwarp_normals(x_nrm, params=p)
            _, rgb_c, dep_c, mask_c, cov = w.warp_rgbd(x_rgb, x_dep, g, a, with_coverage=True)
            _, n_c = w.unwarp_normals(x_nrm, g, a)
            with torch.no_grad():
                planes = w.warp_with_gravity_center_aligned(x_rgb, g, a)
            planes = planes[0] if isinstance(planes, tuple) else planes
            torch.cuda.synchronize()
            for k, t in (("rgb", rgb_w), ("depth", dep_w), ("mask", mask), ("normals", n_hat), ("rgb_call", rgb_c),
                         ("depth_call", dep_c), ("mask_call", mask_c), ("coverage", cov), ("normals_call", n_c), ("planes", planes)):
                out[f"{name}{tag}/{k}"] = _digest(t)
    print(json.dumps(out), flush=True)


def _run(env_extra):
    env = {k: v for k, v in os.environ.items() if not k.startswith("VIDC_")}
    env.update(env_extra)
    res = subprocess.run([sys.executable, os.path.abspath(__file__)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])


@pytest.fixture(scope="module")
def digests(cuda_device):
    return {"off": _run({"VIDC_PF_BULK": "0"}), "default": _run({}), "inverse": _run({"VIDC_INV_PF_WAVES_X100": "8"}),
            "far": _run({"VIDC_INV_PF_WAVES_X100": "100", "VIDC_FWD_PF_WAVES_X100": "100"})}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["default", "inverse", "far"])
def test_bulk_prefetch_keeps_every_bit(digests, variant):
    ref, got = digests["off"], digests[variant]
    assert set(ref) == set(got)
    bad = sorted(k for k in ref if ref[k] != got[k])
    assert not bad, f"{variant}: outputs differ from VIDC_PF_BULK=0: {bad}"


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["off", "default", "inverse"])
def test_unaligned_inputs_without_tensor_maps_keep_every_bit(digests, variant):
    d = digests[variant]
    bad = sorted(k for k in d if "+1/" in k and d[k] != d[k.replace("+1/", "/")])
    assert not bad, f"{variant}: inputs offset by one float differ: {bad}"


if __name__ == "__main__":
    sys.path.insert(0, ROOT)
    _child()
