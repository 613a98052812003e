#!/usr/bin/env python
"""bench.py -- gravity warp+unwarp frames/sec at 640x480 on N B200s, with HBM-roofline accounting.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic frames held by this rank:
    frame parameters (1 CTA / frame) -> fused forward warp of RGB + sparse depth + validity mask
    -> fused inverse warp of the normals with R^T rotation and renormalisation.
Workload (BASELINE.json configs[2], the configuration the metric is quoted on): Azure-Kinect-shaped
640x480 camera, 256 frames per GPU, uniform roll/pitch in +-30 deg, I_a = [0,1,0], seeded synthetic
RGB / dense depth / normals.  Frames are independent: every rank owns its own 256 frames (weak scaling),
there is no data-path collective, NCCL is used for the barrier and the max-over-ranks of the timing only.

Prints ONE JSON line (rank 0).  `value` = frames/s with inputs resident in HBM; `e2e` = the same metric
through the C-ABI host-buffer entry point (pinned host buffers, H2D + kernels + D2H inside the timed
region); `roofline` = dominant kernel against the measured HBM copy bandwidth, every kernel with its own
fraction, the step at the survey's 56 B/px; `cpu_baseline` = the reference's own PyTorch warping executed on the
box's host cores (oracle/_ref, `kind: "reference"`; the C port of it beside, `cpu_port`); `reference_gpu` = the
reference as shipped on one B200 (the "before" number); `dropin` = the unmodified call sequence of
surface_normal.py:148-170 on the drop-in class; `secondary` = the S3 (+-90 deg roll) and S1 (320x240) workloads;
`config5` = BASELINE config 5, the reference's random-init CNNs around the warp, before / after.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from vi_depth_completion_b200 import synthetic as S  # noqa: E402  (seeded synthetic inputs, shared with the tests)

WORKLOAD = "S2"          # 640x480 Azure-Kinect-shaped camera
FRAMES_PER_GPU = 256
BYTES_PER_PX_FWD = 12 + 4 + 12 + 4 + 1   # read RGB+depth, write RGB+depth, write u8 mask
BYTES_PER_PX_INV = 12 + 12               # read normals, write rotated+normalised normals
BYTES_PER_PX_SURVEY = 56                 # SURVEY.md section 8(d): the graded figure (no mask byte)
METRIC = "gravity warp+unwarp frames/sec at 640x480"
UNIT = "frames/s"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """Per-launch DRAM traffic of the dominant kernel from the committed ncu capture, else None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def host_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "samples": len(sm),
                "reasons": sorted(reasons)}


def make_inputs(rank, B):
    cam = S.CAMERAS[WORKLOAD]
    I_g, I_a = S.random_gravity(B, seed=1234 + rank, roll_deg=30.0, pitch_deg=30.0)   # sharding.rank_seed(1234, rank)
    return cam, I_g, I_a


def reference_sequence(w, rgb, depth, normals, g, a):
    """The path exactly as the reference's caller runs it (surface_normal.py:148-170) plus the 3-D depth warp of :110-112:
    warp RGB, warp depth, validity mask, inverse warp + R^T, F.normalize.  `w` is any Warping2DOFAlignment."""
    import torch
    _, x1 = w.warp_with_gravity_center_aligned(rgb, g, a)
    _, d1 = w.warp_with_gravity_center_aligned(depth, g, a)
    mask = (x1[:, 0:1] + x1[:, 1:2] + x1[:, 2:3] > 1e-2).float()
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(normals, g, a)
    return x1, d1, mask, torch.nn.functional.normalize(z, dim=1)


def time_reference_cpu(cam, cores, budget_s, steps=None, warmup=1, log=None):
    """The reference's PyTorch warping path (oracle/_ref, device 'cpu') on `cores` host threads over a bounded sample of the S2
    workload.  Returns the cpu_baseline dict (kind 'reference') or None when the reference files are not on the machine."""
    import torch
    from oracle import ref_loader as RL
    if not RL.reference_available():
        return None
    warnings.filterwarnings("ignore")
    torch.set_num_threads(cores)
    w = RL.load_reference_class("cpu")(*cam)
    H, W = int(w.H), int(w.W)
    I_g, I_a = S.random_gravity(64, seed=1234, roll_deg=30.0, pitch_deg=30.0)
    rgb, depth, normals = S.random_images(64, H, W, seed=1)
    tt = torch.from_numpy

    def run(n):
        t0 = time.perf_counter()
        with torch.no_grad():
            reference_sequence(w, tt(rgb[:n]), tt(depth[:n]), tt(normals[:n]), tt(I_g[:n]), tt(I_a[:n]))
        return time.perf_counter() - t0

    run(1)                                                        # allocator / thread-pool warm-up
    per_frame = run(2) / 2
    n_steps = steps if steps is not None else 3
    sample = int(max(2, min(64, budget_s / max(per_frame * (n_steps + warmup), 1e-6))))
    for _ in range(warmup):
        run(sample)
    times = [run(sample) for _ in range(n_steps)]
    med = float(np.median(times))
    return {"value": sample / med, "unit": UNIT, "cores": cores, "kind": "reference",
            "sample": f"{sample} frames of the S2 workload x {n_steps} timed passes (median) after {warmup} warm-up, the reference's "
                      f"networks/warping_2dof_alignment.py executed on CPU by torch {torch.__version__} with {cores} threads: warp RGB + "
                      "warp depth + mask + inverse warp + F.normalize",
            "ms_per_step": med * 1e3, "frames_per_step": sample, "step_times_s": [round(t, 4) for t in times]}


def time_port_cpu(cam, cores, budget_s, check=None):
    """The C restatement of the reference (oracle/warp_oracle.c, bit-identical to the reference executed on CPU) on `cores`
    pthreads.  `check` = optional (rgb_w, depth_w, mask, normals) host arrays of the GPU run to compare bit for bit."""
    from oracle import oracle as O
    sample = max(2 * cores, 32)
    I_g, I_a = S.random_gravity(FRAMES_PER_GPU, seed=1234, roll_deg=30.0, pitch_deg=30.0)
    orc = O.Oracle(*cam)
    if check is not None:
        s_rgb, s_d, s_n = check["in_rgb"][:sample], check["in_depth"][:sample], check["in_normals"][:sample]
    else:
        s_rgb, s_d, s_n = S.random_images(sample, orc.H, orc.W, seed=1)
        s_d = s_d[:, None]
    O.warp_unwarp_mt(orc, s_rgb[:cores], s_d[:cores], s_n[:cores], I_g[:cores], I_a[:cores], cores)  # warm
    reps, t0 = 0, time.perf_counter()
    while True:
        ref = O.warp_unwarp_mt(orc, s_rgb, s_d, s_n, I_g[:sample], I_a[:sample], cores)
        reps += 1
        if time.perf_counter() - t0 > budget_s or reps >= 50:
            break
    dt = time.perf_counter() - t0
    out = {"value": sample * reps / dt, "unit": UNIT, "cores": cores, "kind": "port",
           "sample": f"{sample} frames x {reps} repetitions of the same step on oracle/warp_oracle.c ({cores} pthreads)"}
    if check is not None:
        out["gpu_output_bit_identical_on_sample"] = bool(
            np.array_equal(ref[0], check["rgb_w"][:sample]) and np.array_equal(ref[2], check["mask"][:sample]) and
            np.array_equal(ref[3], check["normals"][:sample]) and np.array_equal(ref[1], check["depth_w"][:sample, 0]))
    return out


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores -- the reference's PyTorch
    code from oracle/_ref when it travelled here, else the C port of it -- all host threads, a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    cam = S.CAMERAS[WORKLOAD]
    base = time_reference_cpu(cam, cores, budget_s=100.0, steps=max(args.steps, 1), warmup=max(args.warmup, 0))
    port = None
    if base is None:                                             # reference files absent: the port is the arm
        from oracle import oracle as O
        sample = min(256, max(4 * cores, 32))
        I_g, I_a = S.random_gravity(sample, seed=1234, roll_deg=30.0, pitch_deg=30.0)
        orc = O.Oracle(*cam)
        rgb, depth, normals = S.random_images(sample, orc.H, orc.W, seed=1)
        for _ in range(max(args.warmup, 0)):
            O.warp_unwarp_mt(orc, rgb, depth, normals, I_g, I_a, cores)
        times = []
        for _ in range(max(args.steps, 1)):
            t0 = time.perf_counter()
            O.warp_unwarp_mt(orc, rgb, depth, normals, I_g, I_a, cores)
            times.append(time.perf_counter() - t0)
        med = float(np.median(times))
        base = {"value": sample / med, "unit": UNIT, "cores": cores, "kind": "port", "ms_per_step": med * 1e3, "frames_per_step": sample,
                "sample": f"{sample} frames x {len(times)} timed passes (median) after {max(args.warmup, 0)} warm-up, oracle/warp_oracle.c, "
                          f"{cores} pthreads (oracle/_ref absent)"}
    else:
        port = time_port_cpu(cam, cores, budget_s=3.0)
    fps = base["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": base["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{WORKLOAD}: 640x480, {base['frames_per_step']} frames per step (bounded sample of the 256-frame batch), "
                               "warp RGB + warp depth + mask + unwarp normals + renormalise"},
        "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if port is not None:
        line["cpu_port"] = port
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def cuda_time(fn, iters, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def secondary_workloads(dev, iters):
    """BASELINE configs S3 (ScanNet intrinsics, roll in {0, +-45, +-60, +-90} deg) and S1 (320x240, 64 frames): fused step."""
    import torch
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    out = {}
    for name, cam, B, grav in (("S3_extreme_roll_640x480_B256", "S3", 256, "roll"), ("S1_320x240_B64", "S1", 64, "random")):
        w = Warping2DOFAlignment(*S.CAMERAS[cam])
        H, W = int(w.H), int(w.W)
        I_g, I_a = S.extreme_roll_gravity(B, seed=5) if grav == "roll" else S.random_gravity(B, seed=1234)
        g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)
        gen = torch.Generator(device=dev).manual_seed(7)
        rgb = torch.rand(B, 3, H, W, device=dev, generator=gen)
        depth = torch.rand(B, 1, H, W, device=dev, generator=gen) * 9.6 + 0.4
        nrm = torch.randn(B, 3, H, W, device=dev, generator=gen)
        f = cuda_time(lambda: w.warp_rgbd(rgb, depth, g, a), iters)
        i = cuda_time(lambda: w.unwarp_normals(nrm, g, a), iters)
        out[name] = {"forward_ms": f, "inverse_ms": i, "frames_per_s": B / (f + i) * 1e3,
                     "frac_of_hbm_peak_56Bpx": B * H * W * BYTES_PER_PX_SURVEY / (f + i) / 1e6 / measured_peak()[0]}
        del rgb, depth, nrm
    return out


def config5(dev, rank, world, frames_per_gpu=16, steps=3):
    """BASELINE config 5: the reference's SurfaceNormalPrediction + ModifiedFPN (oracle/_ref, unmodified, random init) at 320x240,
    a batch split over the ranks; step time and the share of it spent in the warp / unwarp calls with the reference's own
    warper on the GPU (before) and with the drop-in (after).  None when the reference files are not on the machine."""
    import torch
    from oracle import ref_loader as RL
    if not RL.reference_available():
        return None
    import vi_depth_completion_b200.warping_2dof_alignment as dropin
    warnings.filterwarnings("ignore")
    snp, fpn = RL.ReferenceNetworks(dropin).build(dev, use_mask=False, seed=11)      # INTEGRATION.md section 2 aliasing
    ref_warper = RL.load_reference_class(f"cuda:{dev.index}")(fx=202., fy=202., cx=0.5 * 319.87654, cy=0.5 * 239.87603)
    new_warper = snp.warp_2dof_alignment
    B = frames_per_gpu
    I_g, I_a = S.random_gravity(B, seed=2000 + rank, roll_deg=20, pitch_deg=20)
    rgb = torch.from_numpy(S.smooth_images(B, 240, 320, seed=5 + rank)).to(dev)
    depth = torch.from_numpy(S.random_images(B, 240, 320, seed=6 + rank, sparse_depth=True)[1][:, None]).to(dev)
    g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)
    res = {}
    for tag, warper in (("before_reference_warper", ref_warper), ("after_dropin", new_warper)):
        snp.warp_2dof_alignment = warper
        t_warp = [0.0]

        class Timed:                                             # wall-clock around the two warper calls, GPU synchronised
            def warp_with_gravity_center_aligned(self, *x, **k):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                r = warper.warp_with_gravity_center_aligned(*x, **k)
                torch.cuda.synchronize(); t_warp[0] += time.perf_counter() - t0
                return r

            def inverse_warp_normal_image_with_gravity_center_aligned(self, *x, **k):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                r = warper.inverse_warp_normal_image_with_gravity_center_aligned(*x, **k)
                torch.cuda.synchronize(); t_warp[0] += time.perf_counter() - t0
                return r

        def step():
            with torch.no_grad():
                n = snp(rgb, g, a)                               # main.py:267-269
                return fpn(rgb, n, depth)                        # main.py:274
        step(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        total = (time.perf_counter() - t0) / steps
        snp.warp_2dof_alignment = Timed()
        t_warp[0] = 0.0
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        res[tag] = {"step_ms": total * 1e3, "warp_unwarp_ms": t_warp[0] / steps * 1e3, "warp_share_of_step": (t_warp[0] / steps) / total,
                    "frames_per_s_per_gpu": B / total}
    snp.warp_2dof_alignment = new_warper
    if world > 1:
        import torch.distributed as dist
        for tag in res:
            t = torch.tensor([res[tag]["step_ms"]], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[tag]["step_ms_max_over_ranks"] = float(t.item())
            res[tag]["frames_per_s_aggregate"] = B * world / (float(t.item()) * 1e-3)
    res["frames_per_gpu"] = B
    res["networks"] = "SurfaceNormalPrediction (62.9 M params) + ModifiedFPN (310.3 M params), random init, eval, fp32, 320x240"
    res["speedup_of_the_step"] = res["before_reference_warper"]["step_ms"] / res["after_dropin"]["step_ms"]
    del snp, fpn
    torch.cuda.empty_cache()
    return res


DUMP_FRAMES = 4                 # whole frames written by --dump-outputs (8 planes, 9.8 MB a frame at 640x480)
DUMP_SAMPLE = 1 << 18           # elements of each per-pixel output sampled over the whole batch


def dump_outputs(out_dir, outputs):
    """Writes the outputs of one timed step as out_dir/<name>.npy in float32, about 44 MB in all at 640x480.  Per-frame
    matrices are written in full; each per-pixel output as DUMP_FRAMES whole frames (<name>.npy) and DUMP_SAMPLE elements
    drawn over the whole batch (<name>_sample.npy).  Inputs and choices are seeded, so two builds compare output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    rs = np.random.RandomState(2024)
    for name, t in outputs.items():
        a = t.detach().float()
        if a.dim() == 4:
            frames = np.sort(np.random.RandomState(2023).choice(a.shape[0], min(DUMP_FRAMES, a.shape[0]), replace=False))
            idx = torch.from_numpy(rs.randint(0, a.numel(), size=min(DUMP_SAMPLE, a.numel()))).to(a.device)
            np.save(os.path.join(out_dir, f"{name}_sample.npy"), a.reshape(-1)[idx].cpu().numpy())
            a = a[frames]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from vi_depth_completion_b200 import _cabi, sharding
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = FRAMES_PER_GPU
    cam, I_g, I_a = make_inputs(rank, B)
    w = Warping2DOFAlignment(*cam)
    H, W = int(w.H), int(w.W)
    gen = torch.Generator(device=dev).manual_seed(1 + rank)
    rgb = torch.rand(B, 3, H, W, device=dev, generator=gen)
    depth = torch.rand(B, 1, H, W, device=dev, generator=gen) * 9.6 + 0.4
    normals = torch.randn(B, 3, H, W, device=dev, generator=gen)
    g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)

    lib = _cabi.lib()

    def step():                                # SURVEY.md section 8(d): params kernel + forward kernel + inverse kernel
        p = w.prepare(g, a)               # per-frame parameters, once for the batch
        fwd = w.warp_rgbd(rgb, depth, params=p)      # fused forward (RGB, depth, mask)
        return fwd, w.unwarp_normals(normals, params=p)    # fused inverse (gather, R^T, normalise)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # ---- timed region: EXACTLY K steps, CUDA events on the launching (current) stream ----------
    K = args.steps
    # two events per step inside the timed region (the end of step k is the start of step k+1): an event record between two
    # kernels costs about 5 us of GPU time, so no more of them than the per-kernel split needs
    ev_end = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    ev_mid = [torch.cuda.Event(enable_timing=True) for _ in range(K)]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    launches0 = lib.vidc_launch_count()
    e_start, e_end = ev_end[0], ev_end[K]
    e_start.record()
    for k in range(K):
        # the previous step's outputs go back to the allocator first: the blocks step() used in the warm-up are reused, no
        # allocation from the device inside the timed region; the last step's outputs stay for --dump-outputs
        fwd = inv = None
        p = w.prepare(g, a)
        fwd = w.warp_rgbd(rgb, depth, params=p)
        ev_mid[k].record()
        inv = w.unwarp_normals(normals, params=p)
        ev_end[k + 1].record()
    barrier()
    launches = lib.vidc_launch_count() - launches0
    n_clock_rows_timed = len(sampler.rows) if rank == 0 else 0    # samples taken while the K timed steps ran
    elapsed_ms = e_start.elapsed_time(e_end)
    fwd_ms = float(np.mean([ev_end[k].elapsed_time(ev_mid[k]) for k in range(K)]))
    inv_ms = float(np.mean([ev_mid[k].elapsed_time(ev_end[k + 1]) for k in range(K)]))
    step_ms = [ev_end[k].elapsed_time(ev_end[k + 1]) for k in range(K)]  # SURVEY section 8(d): report median and min too
    # frames are independent: aggregate = sum(frames) / max(elapsed) over ranks, no data-path collective
    _, elapsed_ms, value = sharding.aggregate_throughput(B * K, elapsed_ms, dev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"homography": fwd[0], "rgb_w": fwd[1], "depth_w": fwd[2], "mask": fwd[3], "normals": inv[1]})
    del fwd, inv

    # ---- informational: the same step with the per-frame kernel inside each call (I_g / I_a handed to both entry points) ----
    def step_per_call_params():
        w.warp_rgbd(rgb, depth, g, a)
        w.unwarp_normals(normals, g, a)
    per_call_ms = cuda_time(step_per_call_params, K)
    no_events_ms = cuda_time(step, K)            # the timed step itself, without the per-kernel events inside the loop

    # ---- informational: the opt-in packed layout (channels-last RGBD, one 128-bit load per tap), same frames ----
    packed = torch.cat([rgb, depth], 1).contiguous(memory_format=torch.channels_last)
    packed_ms = cuda_time(lambda: w.warp_rgbd_packed(packed, g, a), K)
    del packed

    # ---- dropin: the UNMODIFIED call sequence of surface_normal.py:148-170 (+ the 3-D depth warp) on the drop-in class -------
    depth3 = depth[:, 0]
    with torch.no_grad():
        dropin_calls = {
            "warp_with_gravity_center_aligned(rgb)": cuda_time(lambda: w.warp_with_gravity_center_aligned(rgb, g, a), K),
            "warp_with_gravity_center_aligned(depth 3-D)": cuda_time(lambda: w.warp_with_gravity_center_aligned(depth3, g, a), K),
            "inverse_warp_normal_image_with_gravity_center_aligned": cuda_time(
                lambda: w.inverse_warp_normal_image_with_gravity_center_aligned(normals, g, a), K),
        }
        dropin_seq_ms = cuda_time(lambda: reference_sequence(w, rgb, depth3, normals, g, a), K)

    # ---- reference_gpu: the reference AS SHIPPED on this B200 (oracle/_ref, 'cuda:N'), same sequence, same 256 frames --------
    reference_gpu = None
    if rank == 0:
        try:
            from oracle import ref_loader as RL
            if RL.reference_available():
                warnings.filterwarnings("ignore")
                rw = RL.load_reference_class(f"cuda:{local}")(*cam)
                with torch.no_grad():
                    reference_sequence(rw, rgb[:2], depth3[:2], normals[:2], g[:2], a[:2])
                    torch.cuda.synchronize()
                    ts = []
                    for _ in range(2):
                        t0 = time.perf_counter()
                        reference_sequence(rw, rgb, depth3, normals, g, a)
                        torch.cuda.synchronize()
                        ts.append(time.perf_counter() - t0)
                reference_gpu = {"value": B / min(ts), "unit": UNIT, "seconds_per_256_frames": min(ts),
                                 "what": "networks/warping_2dof_alignment.py unmodified on cuda (per-sample Python loop, ~45 launches and "
                                         "several host syncs per frame and direction) + the caller's mask and F.normalize",
                                 "dropin_same_sequence_speedup": (B / (dropin_seq_ms * 1e-3)) / (B / min(ts))}
                del rw
        except Exception as e:                                    # the baseline must never take the bench down
            reference_gpu = {"error": repr(e)[:300]}

    # ---- e2e: C-ABI host-buffer entry point, pinned host memory, H2D + kernels + D2H timed --------
    h_rgb = torch.empty(B, 3, H, W, pin_memory=True); h_rgb.copy_(rgb)
    h_depth = torch.empty(B, 1, H, W, pin_memory=True); h_depth.copy_(depth)
    h_nrm = torch.empty(B, 3, H, W, pin_memory=True); h_nrm.copy_(normals)
    h_g = torch.from_numpy(I_g).pin_memory(); h_a = torch.from_numpy(I_a).pin_memory()
    o_rgb = torch.empty(B, 3, H, W, pin_memory=True); o_depth = torch.empty(B, 1, H, W, pin_memory=True)
    o_mask = torch.empty(B, 1, H, W, dtype=torch.uint8, pin_memory=True); o_nrm = torch.empty(B, 3, H, W, pin_memory=True)
    h2d = (h_rgb.numel() + h_depth.numel() + h_nrm.numel() + h_g.numel() + h_a.numel()) * 4
    d2h = (o_rgb.numel() + o_depth.numel() + o_nrm.numel()) * 4 + o_mask.numel()
    stream = torch.cuda.current_stream(dev).cuda_stream

    def e2e_step():
        _cabi.check(lib.vidc_warp_unwarp_host(ctypes.byref(w._cam), B, h_rgb.data_ptr(), h_depth.data_ptr(), h_nrm.data_ptr(),
                                              h_g.data_ptr(), h_a.data_ptr(), o_rgb.data_ptr(), o_depth.data_ptr(),
                                              o_mask.data_ptr(), o_nrm.data_ptr(), ctypes.c_void_p(stream)))

    Ke = max(3, min(K, 10))
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(Ke):
        e2e_step()                  # synchronises its stream before returning
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    _, _, e2e_value = sharding.aggregate_throughput(B * Ke, e2e_s * 1e3, dev)
    clocks = sampler.stop() if rank == 0 else None             # window: timed steps + packed kernel + dropin + e2e steps
    if clocks is not None:
        clocks["samples_during_timed_steps"] = n_clock_rows_timed
    # sanity: the e2e path returns the same bits as the resident path
    _, rgb_w, depth_w, mask = w.warp_rgbd(rgb, depth, g, a)
    torch.cuda.synchronize()
    e2e_ok = bool(torch.equal(rgb_w.cpu(), o_rgb) and torch.equal(mask.cpu(), o_mask))
    del rgb_w, depth_w, mask

    secondary = secondary_workloads(dev, max(5, min(K, 20))) if rank == 0 else None

    # ---- cpu baselines (rank 0, N == 1): the executed reference and its C port on the host cores, bounded samples ----------
    cpu = cpu_port = None
    if rank == 0 and world == 1:
        cores = host_cores()
        check = {"in_rgb": h_rgb.numpy(), "in_depth": h_depth.numpy(), "in_normals": h_nrm.numpy(), "rgb_w": o_rgb.numpy(),
                 "depth_w": o_depth.numpy(), "mask": o_mask.numpy(), "normals": o_nrm.numpy()}
        cpu_port = time_port_cpu(cam, cores, budget_s=8.0, check=check)
        try:
            cpu = time_reference_cpu(cam, cores, budget_s=15.0)
        except Exception as e:
            cpu = None
            cpu_port["reference_error"] = repr(e)[:300]
        if cpu is None:
            cpu, cpu_port = cpu_port, None
    # ---- e2e with the RGB frames as the DataLoader holds them before to_tensor: (B,H,W,3) uint8 (secondary; N == 1) ----------
    e2e_u8 = None
    if rank == 0 and world == 1:
        try:
            gen = torch.Generator().manual_seed(77)
            h_u8 = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, generator=gen).pin_memory()

            def e2e_u8_step():
                _cabi.check(lib.vidc_warp_unwarp_host_u8(ctypes.byref(w._cam), B, h_u8.data_ptr(), h_depth.data_ptr(), h_nrm.data_ptr(),
                                                         h_g.data_ptr(), h_a.data_ptr(), o_rgb.data_ptr(), o_depth.data_ptr(),
                                                         o_mask.data_ptr(), o_nrm.data_ptr(), ctypes.c_void_p(stream)))
            for _ in range(2):
                e2e_u8_step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(Ke):
                e2e_u8_step()
            torch.cuda.synchronize()
            u8_s = time.perf_counter() - t0
            # same bits as the resident float path on ToTensor(frames), checked on the first 8 frames
            x8 = h_u8[:8].permute(0, 3, 1, 2).to(torch.float32).div(255).contiguous().to(dev)
            _, rw8, _, mk8 = w.warp_rgbd(x8, depth[:8], g[:8], a[:8])
            torch.cuda.synchronize()
            e2e_u8 = {"value": B * Ke / u8_s, "unit": UNIT, "h2d_bytes_per_step": h2d - h_rgb.numel() * 4 + h_u8.numel(),
                      "d2h_bytes_per_step": d2h, "steps": Ke,
                      "api": "vidc_warp_unwarp_host_u8 (RGB as (B,H,W,3) uint8 host buffers, ToTensor on the device inside the pipeline)",
                      "matches_resident_path_on_to_tensor": bool(torch.equal(rw8.cpu(), o_rgb[:8]) and torch.equal(mk8.cpu(), o_mask[:8]))}
            del h_u8, x8, rw8, mk8
        except Exception as e:                                    # a secondary number must never take the bench down
            e2e_u8 = {"error": repr(e)[:300]}
    del h_rgb, h_depth, h_nrm, o_rgb, o_depth, o_mask, o_nrm

    # ---- config 5: the reference's CNNs (random init) around the warp, before / after; every rank takes part -------------------
    del rgb, depth, normals
    torch.cuda.empty_cache()
    c5 = None
    try:
        c5 = config5(dev, rank, world)
    except Exception as e:
        c5 = {"error": repr(e)[:300]}

    if rank == 0:
        peak, peak_src = measured_peak()
        px = B * H * W
        # kernel families behind the fused entry points (vidc_kernels.cu: shear_level(), VIDC_SHEAR, default 2)
        shear = os.environ.get("VIDC_SHEAR", "2")[:1]
        fwd_name = "warp_rgbd_fast_kernel" if shear == "0" else "warp_rgbd_shear_kernel"
        inv_name = ("unwarp_normals_box_kernel" if os.environ.get("VIDC_INV_BOX", "0")[:1] == "1" else
                    ("unwarp_normals_shear_kernel" if shear == "2" else "unwarp_normals_fast_kernel"))
        dom = (fwd_name, fwd_ms, BYTES_PER_PX_FWD) if fwd_ms >= inv_ms else (inv_name, inv_ms, BYTES_PER_PX_INV)
        achieved = px * dom[2] / (dom[1] * 1e-3) / 1e9
        traffic = ncu_traffic()

        def kern(ms, bpp):
            gbps = px * bpp / ms / 1e6
            return {"ms": ms, "GBps": gbps, "frac": gbps / peak, "bytes_per_px": bpp}
        per_gpu = value / world
        planes3 = dropin_calls["warp_with_gravity_center_aligned(rgb)"]
        roofline = {"bound": "hbm", "kernel": dom[0], "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": peak_src,
                    "traffic": ((traffic or {}).get(dom[0]) or {}).get("dram_bytes_total"),
                    "traffic_source": ((traffic or {}).get(dom[0]) or {}).get("source"),
                    "algorithmic_bytes_per_launch": px * dom[2],
                    "kernels": {fwd_name: kern(fwd_ms, BYTES_PER_PX_FWD), inv_name: kern(inv_ms, BYTES_PER_PX_INV),
                                "warp_planes_shear_kernel<640,480,3> (the drop-in's RGB warp)": kern(planes3, 24),
                                "warp_rgbd_nhwc4_kernel (opt-in packed RGBD layout, not part of `value`)": kern(packed_ms, BYTES_PER_PX_FWD)},
                    "step": {"bytes_per_frame": H * W * BYTES_PER_PX_SURVEY,
                             "achieved": per_gpu * H * W * BYTES_PER_PX_SURVEY / 1e9,
                             "frac": per_gpu * H * W * BYTES_PER_PX_SURVEY / 1e9 / peak,
                             "bytes_per_px": BYTES_PER_PX_SURVEY,
                             "with_mask_byte": {"bytes_per_px": BYTES_PER_PX_FWD + BYTES_PER_PX_INV,
                                                "frac": per_gpu * H * W * (BYTES_PER_PX_FWD + BYTES_PER_PX_INV) / 1e9 / peak}}}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed_ms / K, "ms_per_step_median": float(np.median(step_ms)), "ms_per_step_min": float(np.min(step_ms)),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{WORKLOAD}: Azure-Kinect-shaped 640x480 (fx=fy=404), {B} frames per GPU, roll/pitch U(-30,30) deg, "
                                   "RGB+depth forward warp + mask, normals inverse warp + R^T + renormalise",
                       "frames_per_gpu": B, "l2": "inputs (2.2 GB per step) larger than L2, no flush needed",
                       "step": "SURVEY 8(d): params kernel + forward kernel + inverse kernel -- prepare(I_g, I_a), warp_rgbd(params=), "
                               "unwarp_normals(params=): 3 launches, nothing cached across steps",
                       "step_with_a_params_kernel_per_call": {"ms_per_step": per_call_ms, "frames_per_s_per_gpu": B / (per_call_ms * 1e-3),
                                                              "launches": 4, "note": "no per-kernel events inside this loop"},
                       "step_without_inner_events": {"ms_per_step": no_events_ms, "frames_per_s_per_gpu": B / (no_events_ms * 1e-3)},
                       "layout": "NCHW fp32", "sharding": f"batch over {world} GPU(s), no data-path collective"},
            "roofline": roofline,
            "cpu_baseline": cpu,
            "cpu_port": cpu_port,
            "reference_gpu": reference_gpu,
            "dropin": {"what": "surface_normal.py:148-170 call sequence unmodified on the drop-in class (+ the 3-D depth warp of :110-112): "
                               "warp RGB, warp depth, the caller's torch mask expression, inverse warp + R^T, the caller's F.normalize",
                       "value": B / (dropin_seq_ms * 1e-3), "unit": UNIT, "ms_per_step": dropin_seq_ms, "ms_per_call": dropin_calls,
                       "frac_of_hbm_peak_56Bpx": B / (dropin_seq_ms * 1e-3) * H * W * BYTES_PER_PX_SURVEY / 1e9 / peak},
            "secondary": secondary,
            "config5": c5,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": Ke, "api": "vidc_warp_unwarp_host (C ABI, pinned host buffers)", "matches_resident_path": e2e_ok},
            "e2e_u8": e2e_u8,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (see dump_outputs; --impl ours only). "
                         "dumps/ in the tree is git-ignored")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
