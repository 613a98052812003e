"""Long random-camera fuzz of the CUDA path against the oracle (a script, not collected by pytest):

    python tests/fuzz_gpu.py [cases=300] [seed=2024]

Random intrinsics (half of the canvases have a width that is a multiple of 32 -> the sheared kernels with the TMA write-out at
run-time geometry; a fifth are the compile-time geometries 640x480 / 320x240 / 640x489 with random focal lengths; the rest take
the straight-row kernels), random batch sizes, moderate / extreme / arbitrary / scaled gravity, white-noise images.  Every
fused entry point, the reference-shaped methods and the prepared-parameter route must land on the oracle's bits."""
import sys, os, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tests import common as C
from tests import exact_reference as X
from oracle import oracle as O
from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment

def main(cases=300, seed=2024):
    O.build()
    dev = torch.device("cuda", 0)
    rs = np.random.RandomState(seed)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    t0 = time.time(); px = 0; paths = {"compile-time": 0, "runtime-sheared": 0, "straight-row": 0}
    for case in range(cases):
        fx = float(rs.uniform(40, 700)); fy = float(fx * rs.uniform(0.9, 1.1))
        u = rs.rand()
        if u < 0.2:
            cx, cy = [(319.87654, 239.87603), (159.93827, 119.938015), (319.529, 244.1902)][rs.randint(3)]; paths["compile-time"] += 1
        elif u < 0.7:
            cx = 16.0 * int(rs.randint(2, 22)) - float(rs.uniform(0.05, 0.45)); cy = float(rs.uniform(15, 260)); paths["runtime-sheared"] += 1
        else:
            cx = float(rs.uniform(20, 340)); cy = float(rs.uniform(15, 260)); paths["straight-row"] += 1
        w, o = Warping2DOFAlignment(fx=fx, fy=fy, cx=cx, cy=cy), O.Oracle(fx, fy, cx, cy)
        assert (int(w.W), int(w.H)) == (o.W, o.H)
        B, kind = int(rs.randint(1, 6)), case % 5
        if kind == 0:
            I_g, I_a = C.random_gravity(B, rs.randint(1 << 30), 30, 30)
        elif kind == 1:
            I_g, I_a = C.random_gravity(B, rs.randint(1 << 30), 89, 80)
        elif kind == 2:
            I_g, I_a = rs.randn(B, 3).astype(np.float32), rs.randn(B, 3).astype(np.float32)
        elif kind == 3:
            I_g, I_a = C.random_gravity(B, rs.randint(1 << 30), 60, 60)
            I_g = (I_g * rs.uniform(0.1, 10, (B, 1))).astype(np.float32)
        else:
            I_g, I_a = C.extreme_roll_gravity(B, rs.randint(1 << 30))
        rgb, depth, nrm = C.random_images(B, o.H, o.W, rs.randint(1 << 30))
        g, a = t(I_g), t(I_a)
        mode = ("bilinear", "nearest")[case % 2]
        _, rgb_w, depth_w, mask, cov = w.warp_rgbd(t(rgb), t(depth), g, a, depth_mode=mode, with_coverage=True)
        _, y = w.warp_with_gravity_center_aligned(t(rgb), g, a)
        _, yd = w.warp_with_gravity_center_aligned(t(depth), g, a, interp_mode=mode)
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(t(nrm), g, a)
        _, nhat, valid = w.unwarp_normals(t(nrm), g, a, with_valid=True)
        p = w.prepare(g, a)
        _, rgb_p, depth_p, mask_p = w.warp_rgbd(t(rgb), t(depth), params=p, depth_mode=mode)
        _, nhat_p = w.unwarp_normals(t(nrm), params=p)
        if o.W % 32 == 0:                                          # channels-last kernels (kernels_shear_cl.cuh): the planar path's bits
            xc = t(rgb).contiguous(memory_format=torch.channels_last); nc = t(nrm).contiguous(memory_format=torch.channels_last)
            _, rgb_c, depth_c, mask_c = w.warp_rgbd(xc, t(depth), g, a, depth_mode=mode)
            _, nhat_c = w.unwarp_normals(nc, g, a)
            _, z_c = w.unwarp_normals(nc, params=p, normalize=False)
            assert torch.equal(rgb_c, rgb_w) and torch.equal(depth_c, depth_w) and torch.equal(mask_c, mask), ("channels-last forward", case)
            assert torch.equal(nhat_c, nhat) and torch.equal(z_c, z), ("channels-last inverse", case)
        with np.errstate(all="ignore"):
            _, oy = o.warp_with_gravity_center_aligned(rgb, I_g, I_a)
            _, oyd = o.warp_with_gravity_center_aligned(depth, I_g, I_a, interp_mode=mode)
            _, oz = o.inverse_warp_normal_image_with_gravity_center_aligned(nrm, I_g, I_a)
            ozn = O.normalize(oz); om = O.validity_mask(oy)
        tag = (case, fx, fy, cx, cy, o.W, o.H, B, kind, mode)
        for name, got, want in (("rgb", rgb_w, oy), ("rgb ref-shaped", y, oy), ("depth", depth_w, oyd), ("depth ref-shaped", yd, oyd),
                                ("unwarp", z, oz), ("unwarp+normalize", nhat, ozn), ("rgb prepared", rgb_p, oy),
                                ("depth prepared", depth_p, oyd), ("unwarp+normalize prepared", nhat_p, ozn)):
            bad = C.count_bit_mismatches(got.cpu().numpy().reshape(want.shape), want)
            assert bad == 0, (name, bad, tag)
        assert np.array_equal(mask.cpu().numpy().reshape(-1), om.reshape(-1)), ("mask", tag)
        assert np.array_equal(mask_p.cpu().numpy().reshape(-1), om.reshape(-1)), ("mask prepared", tag)
        assert np.array_equal(cov.cpu().numpy().astype(np.int64), om.reshape(B, -1).sum(1).astype(np.int64)), ("coverage", tag)
        assert np.array_equal(valid.cpu().numpy().reshape(-1), X.touch_plane(o, I_g, I_a).reshape(-1)), ("valid", tag)
        px += B * o.H * o.W
    print(f"fuzz ok: {cases} cameras, {px / 1e6:.1f} Mpx per output, paths {paths}, {time.time() - t0:.0f} s", flush=True)

if __name__ == "__main__":
    main(*[int(v) for v in sys.argv[1:3]])
