"""Device time of the two backward kernels of the warps, side by side: the atomic scatter (vidc_warp_backward: memset +
scatter) and the fixed-order gather (vidc_warp_backward_ordered).  Development helper, not the bench contract.

    python tools/backward_time.py [iters]

Per workload and kernel: CUDA-event time of one entry-point call (per-frame parameter kernel included) averaged over `iters`
back-to-back calls, the device time of the backward kernel alone from torch.profiler (separate pass), and both as a
fraction of the HBM peak measured in the same run (a 4 GiB device-to-device copy).  Algorithmic bytes: read g (B C H W
fp32) + write grad_in (B C Hin Win fp32), plus the memset of grad_in for the atomic kernel.  S2 and S3 inputs (0.94 GB of g)
exceed the 126 MB L2; S1 (59 MB) fits in it, so its rate is not an HBM figure.
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
from vi_depth_completion_b200._cabi import check, lib  # noqa: E402
from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment, _image, _stream_ptr  # noqa: E402

DEV = torch.device("cuda", 0)
ENTRIES = {"atomic": "vidc_warp_backward", "ordered": "vidc_warp_backward_ordered"}
KERNELS = {"atomic": "warp_backward_kernel", "ordered": "warp_backward_ordered_kernel"}


def hbm_peak_gbs():
    n = 1 << 30                                                   # 4 GiB of fp32, copied device to device
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


def workloads():
    rolls = np.deg2rad(np.where(np.arange(256) % 2 == 0, 90.0, -90.0) + np.random.RandomState(5).uniform(-2, 2, 256))
    g90 = C.gravity_from_angles(rolls.astype(np.float32), np.zeros(256, np.float32))
    a90 = np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (256, 1))
    s2 = C.random_gravity(256, seed=1234, roll_deg=30.0, pitch_deg=30.0)                  # bench.py's S2 frames
    return [("S2_fwd_rgb_B256", "S2", s2, False), ("S2_inv_normals_B256", "S2", s2, True),
            ("S1_fwd_rgb_B64", "S1", C.random_gravity(64, seed=1234), False), ("S1_inv_normals_B64", "S1", C.random_gravity(64, seed=1234), True),
            ("S3_roll90_fwd_rgb_B256", "S3", (g90, a90), False), ("S3_roll90_inv_normals_B256", "S3", (g90, a90), True)]


def main(iters=20):
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = hbm_peak_gbs()
    print(json.dumps({"gpu": smi, "hbm_peak_gbs_measured": round(peak, 1)}), flush=True)
    for name, cam, (I_g, I_a), inverse in workloads():
        w = Warping2DOFAlignment(*C.CAMERAS[cam])
        H, W = int(w.H), int(w.W)
        B = I_g.shape[0]
        g, a = torch.from_numpy(I_g).to(DEV), torch.from_numpy(I_a).to(DEV)
        gout = torch.randn(B, 3, H, W, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
        gi = _image(gout)
        ws = w._params_ws(B, DEV)
        outs = {k: torch.empty((B, 3, H, W), dtype=torch.float32, device=DEV) for k in ENTRIES}

        def call(k):
            check(getattr(lib(), ENTRIES[k])(ctypes.byref(w._cam), ctypes.byref(gi), g.data_ptr(), a.data_ptr(), B, 1 if inverse else 0,
                                              0, ws.data_ptr(), outs[k].data_ptr(), H, W, _stream_ptr(DEV)))

        res = {"workload": name, "B": B, "HxW": f"{H}x{W}"}
        gbytes = B * 3 * H * W * 4
        for k in ENTRIES:
            for _ in range(3):
                call(k)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                call(k)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            nbytes = gbytes * (3 if k == "atomic" else 2)                  # read g, write grad_in (+ memset)
            res[k] = {"call_ms": round(ms, 4), "bytes": nbytes, "call_frac_of_peak": round(nbytes / (ms * 1e-3) / 1e9 / peak, 3)}
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                for k in ENTRIES:
                    call(k)
            torch.cuda.synchronize()
        for k in ENTRIES:
            evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and KERNELS[k] + "<" in e.name]
            kms = sum(e.device_time for e in evs) / max(len(evs), 1) / 1e3
            res[k]["kernel_ms"] = round(kms, 4)
            res[k]["kernel_frac_of_peak"] = round(gbytes * 2 / (kms * 1e-3) / 1e9 / peak, 3) if kms > 0 else None
        diff = (outs["atomic"] - outs["ordered"]).abs().max().item()
        res["max_abs_diff_atomic_vs_ordered"] = diff
        res["ordered_over_atomic_call"] = round(res["ordered"]["call_ms"] / res["atomic"]["call_ms"], 3)
        print(json.dumps(res), flush=True)
        del gout, outs, ws
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 20)
