"""Generates tests/golden/*.npz by EXECUTING the reference (networks/warping_2dof_alignment.py,
normal_utils.py, the mask / renormalise lines of networks/surface_normal.py) on CPU in the build
container.  Run once here; the vectors are committed because /root/reference cannot travel.

    python -m oracle.make_golden

What is frozen
  golden_tiny.npz   64x48 camera, 12 edge-case + 6 random frames: every intermediate and output (H, R, Hinv,
                    both sampler grids, warped RGB, warped depth bilinear / nearest, un-normalised and normalised
                    un-warped normals, validity mask, nearest pyramid masks, loss statistics) IN FULL, except the
                    TINY_DIGESTS arrays, stored like the S configs below so that the file stays under 1 MB.
  golden_demo.npz   BASELINE config 1: the eight demo frames' real gravity + klt tracks through loader code and warper
  golden_tiny_bicubic.npz  64x48, interp_mode='bicubic' outputs IN FULL
  golden_tiny_special.npz  64x48, signed zeros / denormals / inf / NaN inputs: every output IN FULL
  golden_S1/S2/S3.npz  full-resolution configs of SURVEY.md section 8(d): parameters in full, and for the
                    large tensors a SHA-256 of the raw fp32 bytes plus 4096 sampled values (bit-exact check
                    without committing hundreds of MB).
Inputs are regenerated from seeds by tests/common.py (numpy RandomState), so only outputs are stored.
"""
import hashlib
import os
import sys
import warnings

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.ref_loader import REF_ROOT, load_reference_class  # noqa: E402
from tests import common as C  # noqa: E402

warnings.filterwarnings("ignore")
OUT = os.path.join(ROOT, "tests", "golden")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def sample_idx(n, k=4096, seed=99):
    return np.random.RandomState(seed).randint(0, n, size=min(k, n))


def load_normal_utils():
    """normal_utils.py with the undefined `Normalize` bound to F.normalize(x, dim=1) (SURVEY.md Appendix B)."""
    import types
    src = open(os.path.join(REF_ROOT, "normal_utils.py")).read()
    mod = types.ModuleType("reference_normal_utils")
    mod.__dict__["Normalize"] = lambda t: F.normalize(t, dim=1)
    exec(compile(src, "normal_utils.py", "exec"), mod.__dict__)
    return mod


TINY_DIGESTS = ("grid", "inv_grid", "y_rgb", "z")     # the largest, least compressible arrays of golden_tiny.npz


def run_reference(cam_name, I_g, I_a, seed, digest=None):
    """digest: names of the large tensors stored as SHA-256 + samples (None: all of them); the others are stored in full."""
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS[cam_name]
    w = Wref(fx=fx, fy=fy, cx=cx, cy=cy)
    B = I_g.shape[0]
    Hh, Ww = int(w.H), int(w.W)
    rgb, depth, normals = C.random_images(B, Hh, Ww, seed)
    sdepth = C.random_images(B, Hh, Ww, seed, sparse_depth=True)[1]
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    with torch.no_grad():
        H, R, Hi = w._build_homography(g, a)
        Rt, grid, inv_grid = w.image_sampler_forward_inverse(g, a)
        _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
        _, yd = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a)
        _, ydn = w.warp_with_gravity_center_aligned(torch.from_numpy(sdepth), g, a, interp_mode="nearest")
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(normals), g, a)
        zn = F.normalize(z, dim=1)                                            # surface_normal.py:170
        mask = (y[:, 0:1] + y[:, 1:2] + y[:, 2:3] > 1e-2)                     # surface_normal.py:151
        maskf = mask.float()
        pyr = [F.interpolate(maskf, size=s, mode="nearest") for s in ((60, 80), (30, 40), (15, 20), (8, 10))]  # :153-156
        nu = load_normal_utils()
        gt = F.normalize(torch.from_numpy(C.random_images(B, Hh, Ww, seed + 1000)[2]), dim=1)
        loss1, ang1 = nu.compute_normal_vectors_loss_l1(gt, z, maskf)
        loss2, ang2 = nu.compute_normal_vectors_loss_l2(gt, z, maskf)
    out = {"cam": np.array(C.CAMERAS[cam_name], np.float64), "I_g": I_g, "I_a": I_a, "seed": np.int64(seed),
           "W": np.int64(Ww), "H": np.int64(Hh), "K": w.K.numpy(), "K_inv": w.K_inv.numpy(),
           "Hm": H.numpy(), "R": R.numpy(), "Hinv": Hi.numpy(), "Rt_guard": Rt.numpy(),
           "stats": np.array([float(loss1), float(ang1), float(loss2), float(ang2), float(maskf.sum())], np.float64)}
    big = {"grid": grid.numpy(), "inv_grid": inv_grid.numpy(), "y_rgb": y.numpy(), "y_depth": yd.numpy(),
           "y_sdepth_nearest": ydn.numpy(), "z": z.numpy(), "zn": zn.numpy(), "mask": mask.numpy().astype(np.uint8)}
    for i, p in enumerate(pyr):
        big[f"pyr{i}"] = p.numpy().astype(np.uint8)
    for k, v in big.items():
        if digest is not None and k not in digest:
            out[k] = v
            continue
        flat = v.reshape(-1)
        idx = sample_idx(flat.size)
        out[k + "_sha256"] = np.array(sha(v))
        out[k + "_idx"] = idx.astype(np.int64)
        out[k + "_val"] = flat[idx]
        out[k + "_shape"] = np.array(v.shape, np.int64)
    return out


def reference_gravity_rules():
    """The dataset-side gravity conditioning, taken verbatim from the reference source text and executed:
    dataset.py:45-55 (compute_alignment_tensor, ScanNet) and dataset.py:473-483 (Demo loader, identical to :335-345)."""
    import ast
    import textwrap
    src = open(os.path.join(REF_ROOT, "dataset.py")).read()
    lines = src.splitlines()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "compute_alignment_tensor"][0]
    ns = {"torch": torch, "np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "dataset.py", "exec"), ns)
    block = textwrap.dedent("\n".join(lines[472:483]))          # 1-based lines 473..483
    assert block.startswith("gravity_tensor[1] = -gravity_tensor[1]") and "alignment_tensor" in block, block

    def azure(raw):
        loc = {"gravity_tensor": torch.tensor(raw, dtype=torch.float), "torch": torch}
        exec(block, loc)
        return loc["gravity_tensor"].numpy().copy(), loc["alignment_tensor"].numpy().copy()

    def scannet(raw):
        g = torch.tensor(raw, dtype=torch.float)
        return g.numpy().copy(), ns["compute_alignment_tensor"](g).numpy().copy()
    return azure, scannet


def gravity_cases():
    rs = np.random.RandomState(2025)
    raw = rs.randn(512, 3).astype(np.float32)
    raw /= np.linalg.norm(raw, axis=1, keepdims=True).astype(np.float32)
    # near the thresholds: pitch ~ 45 deg (cos 0.707), cos(pitch) ~ 0.3, psi ~ 1e-4 / 1e-6, demo-like vectors
    extra = []
    for p in np.linspace(0.70, 0.72, 41):
        extra.append([0.05, -np.float32(p), -np.float32(np.sqrt(max(0.0, 1 - p * p - 0.0025)))])
    for p in np.linspace(0.29, 0.31, 21):
        extra.append([0.1, np.float32(p), np.float32(np.sqrt(1 - p * p - 0.01))])
    for e in (1e-2, 9.9e-3, 1.01e-2, 1e-3, 7e-4, 0.0):
        extra.append([1.0, np.float32(e), 0.0]); extra.append([1.0, 0.0, -np.float32(e)])
    extra += [[0.09, -0.99, 0.19], [-0.09, -0.99, -0.19], [0.0, -1.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0], [0.0, 0.0, -1.0]]
    return np.concatenate([raw, np.array(extra, np.float32)]).astype(np.float32)


def backward_golden():
    """Row f4: gradients of the executed reference (torch autograd through grid_sample / bmm on CPU)."""
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    w = Wref(fx=fx, fy=fy, cx=cx, cy=cy)
    I_g, I_a = C.random_gravity(6, seed=777, roll_deg=50, pitch_deg=35)
    Hh, Ww = int(w.H), int(w.W)
    rgb, depth, normals = C.random_images(6, Hh, Ww, seed=31)
    wt = np.random.RandomState(5).randn(6, 3, Hh, Ww).astype(np.float32)      # upstream gradient
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    out = {"cam": np.array(C.CAMERAS["tiny"], np.float64), "I_g": I_g, "I_a": I_a, "seed": np.int64(31), "wt_seed": np.int64(5)}
    x = torch.from_numpy(rgb).requires_grad_(True)
    _, y = w.warp_with_gravity_center_aligned(x, g, a)
    (y * torch.from_numpy(wt)).sum().backward()
    out["grad_forward_rgb"] = x.grad.numpy().copy()
    d = torch.from_numpy(depth).requires_grad_(True)
    _, yd = w.warp_with_gravity_center_aligned(d, g, a)
    (yd * torch.from_numpy(wt[:, 0])).sum().backward()
    out["grad_forward_depth"] = d.grad.numpy().copy()
    n = torch.from_numpy(normals).requires_grad_(True)
    _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(n, g, a)
    (z * torch.from_numpy(wt)).sum().backward()
    out["grad_inverse_normals"] = n.grad.numpy().copy()
    n2 = torch.from_numpy(normals).requires_grad_(True)
    _, z2 = w.inverse_warp_normal_image_with_gravity_center_aligned(n2, g, a)
    (F.normalize(z2, dim=1) * torch.from_numpy(wt)).sum().backward()           # through surface_normal.py:170 as well
    out["grad_inverse_normals_normalized"] = n2.grad.numpy().copy()
    return out


def loss_backward_golden():
    """Row a10: the executed reference's normal_utils losses (normal_utils.py:7-34) and their autograd gradients w.r.t.
    pred_normals -- the loss the reference back-propagates at network_run.py:186,248.  Inputs from seeds; pred has four
    channels (only 0:3 are used, :8,:24), some pixels carry exact zeros (norm clamp) and the mask is a sparse 0/1 image."""
    nu = load_normal_utils()
    B, Hh, Ww = 3, 48, 64
    pred, gt, maskf, up = C.loss_inputs(B, Hh, Ww, seed=17)
    out = {"seed": np.int64(17)}
    for name, fn in (("l1", lambda p, g, m: nu.compute_normal_vectors_loss_l1(g, p, m)),
                     ("l1_raw", lambda p, g, m: nu.compute_normal_vectors_loss_l1(g, p, m, normalize_prediction=False)),
                     ("l2", lambda p, g, m: nu.compute_normal_vectors_loss_l2(g, p, m))):
        p = torch.from_numpy(pred).requires_grad_(True)
        loss, angle = fn(p, torch.from_numpy(gt), torch.from_numpy(maskf))
        (loss * float(up)).backward()
        out[f"{name}_loss"] = loss.detach().numpy().copy(); out[f"{name}_angle"] = angle.detach().numpy().copy()
        out[f"{name}_grad"] = p.grad.numpy().copy()
    return out


def rasterize_golden():
    """Row f2: the sparse-depth rasterisation block of the Demo loader (dataset.py:496-510), executed verbatim on synthetic
    tracks (with pixel collisions and out-of-range points) and on the eight demo_dataset track files."""
    import textwrap
    import types
    lines = open(os.path.join(REF_ROOT, "dataset.py")).read().splitlines()
    block = textwrap.dedent("\n".join(lines[495:510]))           # 1-based lines 496..510
    assert block.startswith("klt_depth_tensor = torch.zeros_like(color_tensor[0:1, :, :])") and block.rstrip().endswith("klt_tracks[i, 3]"), block
    fake_self = types.SimpleNamespace(fc=np.array([202.9953, 202.9540]), cc=np.array([159.7645, 122.0951]))

    def run(tracks):
        loc = {"torch": torch, "np": np, "self": fake_self, "color_tensor": torch.zeros(3, 240, 320), "klt_tracks": tracks}
        exec(block, loc)
        return loc["klt_depth_tensor"].numpy().copy()

    rs = np.random.RandomState(77)
    frames = []
    for n in (0, 1, 150, 400):
        z = rs.rand(n) * 3.2 + 0.38
        x = (rs.rand(n) * 2.2 - 1.1) * z
        y = (rs.rand(n) * 1.7 - 0.85) * z
        t = np.stack([np.arange(n, dtype=np.float64), x, y, z, rs.rand(n)], 1) if n else np.zeros((0, 5))
        if n >= 150:                                              # force collisions: repeat a few points with other depths
            t[10:20, 1:3] = t[0:10, 1:3] / t[0:10, 3:4] * t[10:20, 3:4]
        frames.append(t)
    ddir = os.path.join(REF_ROOT, "demo_dataset", "depth_sparse")
    for f in sorted(os.listdir(ddir)):
        frames.append(np.atleast_2d(np.loadtxt(os.path.join(ddir, f), delimiter=" ")))
    N = max(t.shape[0] for t in frames)
    tracks = np.zeros((len(frames), N, 5), np.float64); tracks[:, :, 3] = 1.0
    counts = np.array([t.shape[0] for t in frames], np.int32)
    for i, t in enumerate(frames):
        tracks[i, :t.shape[0], :t.shape[1]] = t
    depth = np.stack([run(t) for t in frames])
    return {"tracks": tracks, "counts": counts, "fc": fake_self.fc, "cc": fake_self.cc, "depth": depth}


def special_values_golden():
    """Signed zeros, denormals, huge values, inf and NaN through the reference (tests/common.py: special_value_images):
    the sign of a zero result, NaN propagation and the out-of-range behaviour of F.normalize, all outputs in full."""
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    w = Wref(fx=fx, fy=fy, cx=cx, cy=cy)
    B, Hh, Ww = 4, int(w.H), int(w.W)
    rgb, depth, normals = C.special_value_images(B, Hh, Ww, seed=21)
    I_g, I_a = C.special_value_gravity(B)
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    with torch.no_grad():
        _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
        _, yd = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a)
        _, ydn = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a, interp_mode="nearest")
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(normals), g, a)
        zn = F.normalize(z, dim=1)
        mask = (y[:, 0:1] + y[:, 1:2] + y[:, 2:3] > 1e-2)
    return {"B": np.int64(B), "seed": np.int64(21), "I_g": I_g, "I_a": I_a, "y_rgb": y.numpy(), "y_depth": yd.numpy(),
            "y_depth_nearest": ydn.numpy(), "z": z.numpy(), "zn": zn.numpy(), "mask": mask.numpy().astype(np.uint8)}


def bicubic_golden():
    """interp_mode='bicubic' through the reference (valid in F.grid_sample, never used by the reference's callers): the 64x48
    camera, edge-case + random gravity, RGB and the 3-D depth path, all outputs in full."""
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["tiny"]
    w = Wref(fx=fx, fy=fy, cx=cx, cy=cy)
    eg, ea = C.edge_case_gravity()
    rg, ra = C.random_gravity(6, seed=4321, roll_deg=60, pitch_deg=45)
    I_g, I_a = np.concatenate([eg, rg]), np.concatenate([ea, ra])
    B, Hh, Ww = I_g.shape[0], int(w.H), int(w.W)
    rgb, depth, _ = C.random_images(B, Hh, Ww, seed=7)
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    with torch.no_grad():
        _, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a, interp_mode="bicubic")
        _, yd = w.warp_with_gravity_center_aligned(torch.from_numpy(depth), g, a, interp_mode="bicubic")
    return {"I_g": I_g, "I_a": I_a, "seed": np.int64(7), "y_rgb": y.numpy(), "y_depth": yd.numpy()}


def demo_golden():
    """BASELINE config 1 without the PNGs: the eight demo_dataset frames' REAL gravity files and klt track files through the
    reference's own loader code (gravity conditioning dataset.py:473-483, rasterisation :496-510) and warper (S1 intrinsics,
    main.py:243), with seeded smooth synthetic RGB standing in for the colour images and seeded random normals for the
    CNN output.  Small inputs in full, the large outputs as SHA-256 + 4096 samples."""
    Wref = load_reference_class("cpu")
    fx, fy, cx, cy = C.CAMERAS["S1"]
    w = Wref(fx=fx, fy=fy, cx=cx, cy=cy)
    gdir = os.path.join(REF_ROOT, "demo_dataset", "gravity")
    raw = np.stack([np.loadtxt(os.path.join(gdir, f)).astype(np.float32) for f in sorted(os.listdir(gdir))])   # dataset.py:472
    azure, _ = reference_gravity_rules()
    cond = [azure(r) for r in raw]
    I_g, I_a = np.stack([c[0] for c in cond]), np.stack([c[1] for c in cond])
    ras = rasterize_golden()
    tracks, counts, depth = ras["tracks"][-8:], ras["counts"][-8:], ras["depth"][-8:]          # the eight demo track files
    B, Hh, Ww = 8, int(w.H), int(w.W)
    rgb = C.smooth_images(B, Hh, Ww, seed=11)
    normals = C.random_images(B, Hh, Ww, seed=12)[2]
    g, a = torch.from_numpy(I_g), torch.from_numpy(I_a)
    with torch.no_grad():
        H, y = w.warp_with_gravity_center_aligned(torch.from_numpy(rgb), g, a)
        _, yd = w.warp_with_gravity_center_aligned(torch.from_numpy(depth[:, 0]), g, a)
        _, ydn = w.warp_with_gravity_center_aligned(torch.from_numpy(depth[:, 0]), g, a, interp_mode="nearest")
        mask = (y[:, 0:1] + y[:, 1:2] + y[:, 2:3] > 1e-2)
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(torch.from_numpy(normals), g, a)
        zn = F.normalize(z, dim=1)
    out = {"raw_gravity": raw, "I_g": I_g, "I_a": I_a, "tracks": tracks, "counts": counts, "fc": ras["fc"], "cc": ras["cc"],
           "Hm": H.numpy(), "rgb_seed": np.int64(11), "normals_seed": np.int64(12),
           "valid_fraction": np.float64(mask.float().mean())}
    for k, v in {"depth": depth, "y_rgb": y.numpy(), "y_depth": yd.numpy(), "y_depth_nearest": ydn.numpy(),
                 "mask": mask.numpy().astype(np.uint8), "zn": zn.numpy()}.items():
        flat = v.reshape(-1)
        idx = sample_idx(flat.size)
        out[k + "_sha256"] = np.array(sha(v)); out[k + "_idx"] = idx.astype(np.int64); out[k + "_val"] = flat[idx]
        out[k + "_shape"] = np.array(v.shape, np.int64)
    return out


def main():
    os.makedirs(OUT, exist_ok=True)
    if "--only-loss-backward" in sys.argv:
        np.savez_compressed(os.path.join(OUT, "golden_tiny_loss_backward.npz"), **loss_backward_golden())
        return
    np.savez_compressed(os.path.join(OUT, "golden_tiny_loss_backward.npz"), **loss_backward_golden())
    # tiny: edge cases + random, everything but TINY_DIGESTS in full
    eg, ea = C.edge_case_gravity()
    rg, ra = C.random_gravity(6, seed=4321, roll_deg=60, pitch_deg=45)
    np.savez_compressed(os.path.join(OUT, "golden_tiny.npz"),
                        **run_reference("tiny", np.concatenate([eg, rg]), np.concatenate([ea, ra]), seed=7, digest=TINY_DIGESTS))
    # full-resolution configs: digests
    for name, (B, roll, pitch, seed) in {"S1": (6, 30, 30, 1), "S2": (3, 30, 30, 2), "S3": (3, 75, 40, 3)}.items():
        I_g, I_a = C.random_gravity(B, seed=1234, roll_deg=roll, pitch_deg=pitch)
        if name == "S3":
            xg, xa = C.extreme_roll_gravity(3, seed=5)
            I_g, I_a = np.concatenate([I_g, xg]), np.concatenate([I_a, xa])
        np.savez_compressed(os.path.join(OUT, f"golden_{name}.npz"), **run_reference(name, I_g, I_a, seed))
    np.savez_compressed(os.path.join(OUT, "golden_tiny_backward.npz"), **backward_golden())
    np.savez_compressed(os.path.join(OUT, "golden_rasterize.npz"), **rasterize_golden())
    np.savez_compressed(os.path.join(OUT, "golden_tiny_special.npz"), **special_values_golden())
    np.savez_compressed(os.path.join(OUT, "golden_tiny_bicubic.npz"), **bicubic_golden())
    np.savez_compressed(os.path.join(OUT, "golden_demo.npz"), **demo_golden())
    raw = gravity_cases()
    azure, scannet = reference_gravity_rules()
    ga = [azure(r) for r in raw]; gs = [scannet(r) for r in raw]
    np.savez_compressed(os.path.join(OUT, "golden_gravity.npz"), raw=raw,
                        azure_g=np.stack([x[0] for x in ga]), azure_a=np.stack([x[1] for x in ga]),
                        scannet_g=np.stack([x[0] for x in gs]), scannet_a=np.stack([x[1] for x in gs]))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
