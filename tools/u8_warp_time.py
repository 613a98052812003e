"""Device time of the fused uint8 forward warp (warp_rgbd_u8) against the two passes it replaces (to_tensor_u8, then
warp_rgbd), both with a prepared workspace (params=), on the same frames in one process.  Development helper, not the bench
contract.

    python tools/u8_warp_time.py [rounds] [iters]

Workloads: S2 (640x480, 256 frames, roll / pitch in +-30 deg), S3 (ScanNet intrinsics, 256 frames all at one roll: 0, +-45,
+-90 deg) and S1 (320x240, 64 frames).  Per workload:
  * call time: CUDA events around `iters` calls, the two routes alternating for `rounds` rounds (min and max per route, and
    whether the fused route was faster in every round);
  * kernel time: the device durations torch.profiler records for the same calls, in a pass of its own;
  * fraction of the HBM peak: the fused route's 24 B/px (3 B of RGB and 4 B of depth read; 12 B of RGB, 4 B of depth and
    1 B of mask written) over its kernel time, against a 4 GiB device copy measured in the same run.  The two-pass route
    moves 48 B/px (to_tensor: 3 + 12; the warp: 12 + 4 + 12 + 4 + 1).
  * the outputs of both routes, compared bit for bit.
The S2 / S3 frames (236 MB of uint8, 943 MB as float) exceed the 126 MB L2; S1 at 64 frames (15 MB + 20 MB) does not.
"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.autograd import DeviceType  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from vi_depth_completion_b200 import synthetic as S  # noqa: E402
from vi_depth_completion_b200.gravity import to_tensor_u8  # noqa: E402
from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment  # noqa: E402

DEV = torch.device("cuda", 0)
FUSED_BPP, TWO_PASS_BPP = 24, 48


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
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_ms(fn, iters):
    """Mean device time per call of the kernels fn launches (torch.profiler, CUDA activity)."""
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset")):
            name = e.name.split("(")[0].removeprefix("void ").removeprefix("vidc_k::")
            per[name] = per.get(name, 0.0) + e.device_time / 1e3 / iters
    return sum(per.values()), {k: round(v, 4) for k, v in per.items()}


def same_bits(x, y):
    x, y = x.contiguous(), y.contiguous()
    if x.dtype == torch.float32:
        x, y = x.view(torch.int32), y.view(torch.int32)
    return x.shape == y.shape and bool(torch.equal(x, y))


def workload(name, cam, I_g, I_a, peak, rounds, iters):
    w = Warping2DOFAlignment(*S.CAMERAS[cam])
    B, H, W = I_g.shape[0], int(w.H), int(w.W)
    gen = torch.Generator(device=DEV).manual_seed(7)
    u8 = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=DEV, generator=gen)
    depth = torch.rand(B, 1, H, W, device=DEV, generator=gen) * 9.6 + 0.4
    p = w.prepare(torch.from_numpy(I_g).to(DEV), torch.from_numpy(I_a).to(DEV))
    two_pass = lambda: w.warp_rgbd(to_tensor_u8(u8), depth, params=p)
    fused = lambda: w.warp_rgbd_u8(u8, depth, params=p)
    with torch.no_grad():
        a, b = two_pass(), fused()
        torch.cuda.synchronize()
        identical = all(same_bits(x, y) for x, y in zip(a[1:], b[1:]))
        del a, b
        for _ in range(3):
            two_pass(); fused()
        t2, tf = [], []
        for _ in range(rounds):                                    # alternating: each round times both routes
            t2.append(timed(two_pass, iters))
            tf.append(timed(fused, iters))
        k2, k2_parts = kernel_ms(two_pass, iters)
        kf, kf_parts = kernel_ms(fused, iters)
    px = B * H * W
    return {"workload": name, "frames": B, "canvas": f"{W}x{H}", "bit_identical": identical,
            "two_pass_call_ms": [round(min(t2), 4), round(max(t2), 4)], "fused_call_ms": [round(min(tf), 4), round(max(tf), 4)],
            "fused_faster_every_round": all(f < t for f, t in zip(tf, t2)),
            "call_speedup_min_ratio": round(min(t2) / min(tf), 3),
            "two_pass_kernel_ms": round(k2, 4), "fused_kernel_ms": round(kf, 4), "kernels": {**k2_parts, **kf_parts},
            "fused_frac_of_peak_24Bpx": round(px * FUSED_BPP / (kf * 1e-3) / 1e9 / peak, 3),
            "two_pass_frac_of_peak_48Bpx": round(px * TWO_PASS_BPP / (k2 * 1e-3) / 1e9 / peak, 3)}


def main(rounds=7, iters=20):
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = hbm_peak_gbs()
    print(json.dumps({"gpu": smi, "hbm_peak_gbs_measured": round(peak, 1), "rounds": rounds, "iters": iters}), flush=True)
    runs = [("S2_640x480_B256", "S2", S.random_gravity(256, seed=1234, roll_deg=30.0, pitch_deg=30.0))]
    for roll in (0, 45, -45, 90, -90):
        g = S.gravity_from_angles(np.full(256, np.deg2rad(roll), np.float32), np.zeros(256, np.float32))
        runs.append((f"S3_roll{roll:+d}_B256", "S3", (g, np.tile(np.array([[0.0, 1.0, 0.0]], np.float32), (256, 1)))))
    runs.append(("S1_320x240_B64", "S1", S.random_gravity(64, seed=1234)))
    for name, cam, (I_g, I_a) in runs:
        print(json.dumps(workload(name, cam, I_g, I_a, peak, rounds, iters)), flush=True)
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main(*(int(a) for a in sys.argv[1:3]))
