"""A/B timing of the sheared kernels' L2 prefetch forms (kernels_shear.cuh), one build, fresh processes.

    python tools/prefetch_time.py [--rounds 5] [--steps 200] [--sweep-rounds 2]

1. bench.py --gpus 1 --steps STEPS in fresh processes, the variants alternating ROUNDS times:
     base       VIDC_PF_BULK=0 (per-thread forward prefetch, no inverse prefetch)
     bulk_fwd   bulk forward prefetch, no inverse prefetch (VIDC_INV_PF_WAVES_X100=0)
     bulk_both  bulk forward + inverse prefetch (the default)
   prints median and spread (max - min) of `value`, of the forward and inverse kernel times in the step and of the S3 / S1
   secondary figures.
2. a distance sweep (forward and inverse, percent of a wave of resident CTAs): the bench step (prepare + fused forward + fused
   inverse, S2, 256 frames) timed with CUDA events in a fresh process per point (--inner), the points alternating.
The card's name and power limit are read in the same call.  Writes nothing but stdout.
The base arm is the per-thread form compiled in this build.  It runs slower than the same form did before the bulk form was
added (profiles/r4_history.md), so judge a change against the previous commit built alongside, not against this arm.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = {
    "base": {"VIDC_PF_BULK": "0"},
    "bulk_fwd": {"VIDC_INV_PF_WAVES_X100": "0"},
    "bulk_both": {},
}
SWEEP = [("inv", v) for v in (0, 4, 16, 50)] + [("fwd", v) for v in (2, 16)] + [("base", 0)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                     # informational only
        return repr(e)


def run(cmd, env_extra):
    env = dict(os.environ, **env_extra)
    res = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    for line in reversed(res.stdout.splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError(f"{cmd} {env_extra}: no JSON line\n{res.stdout[-2000:]}\n{res.stderr[-2000:]}")


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2] if len(xs) % 2 else 0.5 * (xs[len(xs) // 2 - 1] + xs[len(xs) // 2]),
            "spread": xs[-1] - xs[0], "n": len(xs), "all": xs}


def inner(steps):
    """The bench step at the bench workload, CUDA events around `steps` steps (after warm-up): forward, inverse, step ms."""
    import numpy as np
    import torch
    import bench
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    dev = torch.device("cuda", 0)
    B = bench.FRAMES_PER_GPU
    cam, I_g, I_a = bench.make_inputs(0, B)
    w = Warping2DOFAlignment(*cam)
    H, W = int(w.H), int(w.W)
    gen = torch.Generator(device=dev).manual_seed(1)
    rgb = torch.rand(B, 3, H, W, device=dev, generator=gen)
    depth = torch.rand(B, 1, H, W, device=dev, generator=gen) * 9.6 + 0.4
    normals = torch.randn(B, 3, H, W, device=dev, generator=gen)
    g, a = torch.from_numpy(I_g).to(dev), torch.from_numpy(I_a).to(dev)
    for _ in range(5):
        p = w.prepare(g, a)
        w.warp_rgbd(rgb, depth, params=p)
        w.unwarp_normals(normals, params=p)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * steps)]
    for k in range(steps):
        p = w.prepare(g, a)
        ev[3 * k].record()
        w.warp_rgbd(rgb, depth, params=p)
        ev[3 * k + 1].record()
        w.unwarp_normals(normals, params=p)
        ev[3 * k + 2].record()
    torch.cuda.synchronize()
    fwd = float(np.median([ev[3 * k].elapsed_time(ev[3 * k + 1]) for k in range(steps)]))
    inv = float(np.median([ev[3 * k + 1].elapsed_time(ev[3 * k + 2]) for k in range(steps)]))
    print(json.dumps({"forward_ms": fwd, "inverse_ms": inv}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--sweep-rounds", type=int, default=2)
    ap.add_argument("--inner", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.inner:
        return inner(args.steps)
    from vi_depth_completion_b200 import build as vb
    vb.build()
    vb.build_torch_ops()
    print("card:", card(), flush=True)

    res = {k: {"value": [], "forward_ms": [], "inverse_ms": [], "S3_frames_per_s": [], "S1_frames_per_s": []} for k in VARIANTS}
    for r in range(args.rounds):
        for name, env in VARIANTS.items():
            j = run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", "10"], env)
            kern = j["roofline"]["kernels"]
            res[name]["value"].append(j["value"])
            res[name]["forward_ms"].append(kern["warp_rgbd_shear_kernel"]["ms"])
            res[name]["inverse_ms"].append(kern["unwarp_normals_shear_kernel"]["ms"])
            res[name]["S3_frames_per_s"].append(j["secondary"]["S3_extreme_roll_640x480_B256"]["frames_per_s"])
            res[name]["S1_frames_per_s"].append(j["secondary"]["S1_320x240_B64"]["frames_per_s"])
            print(f"round {r} {name}: value {j['value']:.1f}  fwd {res[name]['forward_ms'][-1]:.4f} ms  "
                  f"inv {res[name]['inverse_ms'][-1]:.4f} ms", flush=True)
    summary = {name: {k: stats(v) for k, v in d.items()} for name, d in res.items()}
    print(json.dumps({"bench_ab": summary}), flush=True)
    base = summary["base"]["value"]["median"]
    for name in VARIANTS:
        s = summary[name]
        print(f"{name:10s} value {s['value']['median']:10.1f} (spread {s['value']['spread']:7.1f}, {100 * (s['value']['median'] / base - 1):+.2f} %)"
              f"  fwd {s['forward_ms']['median']:.4f}  inv {s['inverse_ms']['median']:.4f} ms"
              f"  S3 {s['S3_frames_per_s']['median']:.0f}  S1 {s['S1_frames_per_s']['median']:.0f} frames/s", flush=True)

    sweep = {f"{k}{v}": {"forward_ms": [], "inverse_ms": []} for k, v in SWEEP}
    for r in range(args.sweep_rounds):
        for kind, v in SWEEP:
            env = ({"VIDC_PF_BULK": "0"} if kind == "base" else
                   {"VIDC_INV_PF_WAVES_X100": str(v)} if kind == "inv" else {"VIDC_FWD_PF_WAVES_X100": str(v)})
            j = run([sys.executable, os.path.abspath(__file__), "--inner", "--steps", "100"], env)
            for k in ("forward_ms", "inverse_ms"):
                sweep[f"{kind}{v}"][k].append(j[k])
    print(json.dumps({"sweep": {k: {m: stats(x) for m, x in d.items()} for k, d in sweep.items()}}), flush=True)
    for k, d in sweep.items():
        print(f"{k:8s} fwd {stats(d['forward_ms'])['median']:.4f}  inv {stats(d['inverse_ms'])['median']:.4f} ms", flush=True)
    print("card:", card(), flush=True)


if __name__ == "__main__":
    main()
