"""Device time of the gravity gradient: vidc_warp_backward_params (per-frame parameter kernel, the per-tile partial sums and
the tile reduction) followed by vidc_frame_params_backward, next to the image backward (vidc_warp_backward) of the same
workload and to torch's autograd of the fp32 restatement (tests/gravity_grad_reference.py) on the same GPU -- what a caller
had to run before.  Development helper, not the bench contract.

    python tools/gravity_grad_time.py [iters]

Algorithmic bytes of the parameter gradient: per output pixel the four taps of x and the upstream gradient, 4 + 1 floats per
channel (about 24 B/px for one channel, 60 B/px for three), against the HBM peak measured in the same run (a 4 GiB copy).
The S2 inputs (0.94 GB per tensor) exceed the 126 MB L2; S1 at B = 64 (59 MB) fits in it, so its rate is not an HBM figure.
"""
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests import common as C  # noqa: E402
from tests import gravity_grad_reference as GR  # noqa: E402
from vi_depth_completion_b200 import _cabi  # noqa: E402
from vi_depth_completion_b200._cabi import check, lib  # noqa: E402
from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment, _image, _stream_ptr  # noqa: E402

DEV = torch.device("cuda", 0)


def hbm_peak_gbs():
    n = 1 << 30
    src = torch.empty(n, dtype=torch.float32, device=DEV).fill_(1.0)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * 4 * n * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del src, dst
    torch.cuda.empty_cache()
    return gbs


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main(iters=20):
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = hbm_peak_gbs()
    print(json.dumps({"gpu": smi, "hbm_peak_gbs_measured": round(peak, 1)}), flush=True)
    s2 = C.random_gravity(256, seed=1234, roll_deg=30.0, pitch_deg=30.0)
    s1 = C.random_gravity(64, seed=1234)
    for name, cam, (I_g, I_a), inverse in (("S2_fwd_rgb_B256", "S2", s2, False), ("S2_inv_normals_B256", "S2", s2, True),
                                           ("S1_fwd_rgb_B64", "S1", s1, False), ("S1_inv_normals_B64", "S1", s1, True)):
        w = Warping2DOFAlignment(*C.CAMERAS[cam])
        H, W = int(w.H), int(w.W)
        B = I_g.shape[0]
        g, a = torch.from_numpy(I_g).to(DEV), torch.from_numpy(I_a).to(DEV)
        gen = torch.Generator(device=DEV).manual_seed(1)
        x = torch.rand(B, 3, H, W, device=DEV, generator=gen)
        gout = torch.randn(B, 3, H, W, device=DEV, generator=gen)
        xi, gi = _image(x), _image(gout)
        ws = w._params_ws(B, DEV)
        scratch = torch.empty(int(lib().vidc_warp_backward_params_scratch_bytes(ctypes.byref(w._cam), B)) // 8, dtype=torch.float64, device=DEV)
        gp = torch.empty((B, _cabi.FRAME_PARAMS_FLOATS), dtype=torch.float32, device=DEV)
        gg, ga = torch.empty_like(g), torch.empty_like(a)
        gx = torch.empty((B, 3, H, W), dtype=torch.float32, device=DEV)

        def params_grad():
            check(lib().vidc_warp_backward_params(ctypes.byref(w._cam), ctypes.byref(xi), ctypes.byref(gi), g.data_ptr(), a.data_ptr(), B,
                                                  1 if inverse else 0, 0, ws.data_ptr(), scratch.data_ptr(), gp.data_ptr(), _stream_ptr(DEV)))
            check(lib().vidc_frame_params_backward(ctypes.byref(w._cam), g.data_ptr(), a.data_ptr(), B, gp.data_ptr(), None, gg.data_ptr(),
                                                   ga.data_ptr(), _stream_ptr(DEV)))

        def image_grad():
            check(lib().vidc_warp_backward(ctypes.byref(w._cam), ctypes.byref(gi), g.data_ptr(), a.data_ptr(), B, 1 if inverse else 0, 0,
                                           ws.data_ptr(), gx.data_ptr(), H, W, _stream_ptr(DEV)))

        res = {"workload": name, "B": B, "HxW": f"{H}x{W}"}
        nbytes = B * H * W * 3 * (4 + 1) * 4
        ms = timed(params_grad, iters)
        res["gravity_grad"] = {"call_ms": round(ms, 4), "bytes": nbytes, "frac_of_peak": round(nbytes / (ms * 1e-3) / 1e9 / peak, 3)}
        res["image_grad_atomic_call_ms"] = round(timed(image_grad, iters), 4)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                params_grad()
            torch.cuda.synchronize()
        for k in ("warp_grad_params_kernel", "grad_params_reduce_kernel", "frame_params_backward_kernel"):
            evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and k in e.name]
            res[k + "_ms"] = round(sum(e.device_time for e in evs) / max(len(evs), 1) / 1e3, 4)

        # before: torch autograd of the fp32 restatement on the same GPU (parameters on the host, as the reference's loops are)
        cam32 = GR.Camera(w._cam, torch.float32)
        cam32.K, cam32.K_inv, cam32.corners = cam32.K.to(DEV), cam32.K_inv.to(DEV), cam32.corners.to(DEV)

        def torch_autograd():
            gr, ar = g.clone().requires_grad_(True), a.clone().requires_grad_(True)
            p = GR.build_homography(cam32, gr, ar)
            sc = GR.frame_scale(cam32, p[0])
            prm = dict(sc, H=p[0], R=p[1], Hinv=p[2])
            grid = (GR.inverse_grid if inverse else GR.forward_grid)(cam32, {k: v for k, v in prm.items()})
            y = torch.nn.functional.grid_sample(x, grid, mode="bilinear", padding_mode="zeros", align_corners=False)
            if inverse:
                y = torch.bmm(prm["R"].transpose(1, 2), y.reshape(B, 3, -1))
            y.backward(gout.reshape(y.shape))
        try:
            res["torch_fp32_restatement_autograd_ms"] = round(timed(torch_autograd, max(iters // 10, 2)), 3)
        except Exception as e:                      # noqa: BLE001 -- report, keep the kernel numbers
            res["torch_fp32_restatement_autograd_ms"] = f"failed: {type(e).__name__}: {e}"
        print(json.dumps(res), flush=True)
        del x, gout, gx, scratch
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 20)
