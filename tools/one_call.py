import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, numpy as np
from tests import common as C
from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
cam = sys.argv[1] if len(sys.argv) > 1 else "S1"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 2
dev = torch.device("cuda", 0)
w = Warping2DOFAlignment(*C.CAMERAS[cam]); H, W = int(w.H), int(w.W)
I_g, I_a = C.random_gravity(B, 1234)
rgb, depth, nrm = C.random_images(B, H, W, 1)
t = lambda x: torch.from_numpy(x).to(dev)
out = w.warp_rgbd(t(rgb), t(depth), t(I_g), t(I_a))
torch.cuda.synchronize()
print("ok", float(out[1].sum()))
# one backward call of each variant (atomic scatter, fixed-order gather), forward and inverse warp, bilinear and nearest
for det in (False, True):
    w.deterministic_backward = det
    for mode in ("bilinear", "nearest"):
        x = t(rgb).requires_grad_(True)
        w.warp_with_gravity_center_aligned(x, t(I_g), t(I_a), interp_mode=mode)[1].sum().backward()
        torch.cuda.synchronize()
        print("backward", "ordered" if det else "atomic", mode, float(x.grad.sum()))
    n = t(nrm).requires_grad_(True)
    w.inverse_warp_normal_image_with_gravity_center_aligned(n, t(I_g), t(I_a))[1].sum().backward()
    torch.cuda.synchronize()
    print("backward", "ordered" if det else "atomic", "inverse", float(n.grad.sum()))
