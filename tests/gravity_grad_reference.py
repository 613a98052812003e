"""Plain-torch, differentiable restatement of the reference's parameter chain and warps (SURVEY.md Appendix A.1-A.5, plus the
bmm with R^T of the inverse warp), for the gravity gradient.

TEST INFRASTRUCTURE ONLY.  Every function uses the torch op the reference uses at the cited line of
networks/warping_2dof_alignment.py, so torch's autograd of these functions is the reference's autograd.  `dtype` selects the
precision: float32 is the reference as torch runs it, float64 the truth the CUDA gradients are measured against.  The camera
constants (K, K^-1, the fp32 principal point and 1 / (W / 2)) are the fp32 values the reference stores, in either dtype.
"""
import numpy as np
import torch
import torch.nn.functional as F

FIELDS = ("H", "R", "Hinv", "px_min", "py_min", "kw", "kh", "ikw", "ikh", "w_max", "h_max")


class Camera:
    """The reference's constants (:6-24) as torch tensors of `dtype`, from a vidc_camera."""

    def __init__(self, cam, dtype=torch.float64):
        self.W, self.H = int(cam.W), int(cam.H)
        self.dtype = dtype
        self.K = torch.tensor(np.array(cam.K, np.float32).reshape(3, 3), dtype=dtype)
        self.K_inv = torch.tensor(np.array(cam.Kinv, np.float32).reshape(3, 3), dtype=dtype)
        self.cx, self.cy = float(np.float32(cam.cx)), float(np.float32(cam.cy))
        self.ihw, self.ihh = float(np.float32(cam.inv_half_w)), float(np.float32(cam.inv_half_h))
        W, H = self.W, self.H
        # :18 -- np.array([...]).transpose(): a column-major (3,4) operand
        self.corners = torch.tensor(np.array([[0, 0, 1], [W - 1, 0, 1], [0, H - 1, 1], [W - 1, H - 1, 1]], np.float32),
                                    dtype=dtype).t()


def _skew(v):
    """[v]x of a (B,3) tensor (:26-32)."""
    z = torch.zeros_like(v[:, 0])
    return torch.stack([torch.stack([z, -v[:, 2], v[:, 1]], 1), torch.stack([v[:, 2], z, -v[:, 0]], 1),
                        torch.stack([-v[:, 1], v[:, 0], z], 1)], 1)


def build_homography(cam, I_g, I_a):
    """:35-58 -> (H, R, Hinv), each (B,3,3)."""
    B = I_g.shape[0]
    g, a = I_g.reshape(B, 3, 1), I_a.reshape(B, 3)
    q = torch.bmm(-_skew(a), g)                                  # :41-42  q = (-[a]x) g
    d = torch.bmm(a.reshape(B, 1, 3), g).reshape(B, 1)           # :43
    n = q.reshape(B, 3).norm(dim=1, keepdim=True)                # :44
    q4 = torch.cos(0.5 * torch.atan2(n, d))                      # :48
    q = q.reshape(B, 3) / (2.0 * q4)                             # :51
    S = _skew(q)                                                 # :52
    I3 = torch.eye(3, dtype=I_g.dtype, device=I_g.device)
    R = (I3 + (2.0 * q4).reshape(B, 1, 1) * S) + 2.0 * torch.matmul(S, S)   # :53-54
    H = torch.matmul(torch.matmul(cam.K, R), cam.K_inv)          # :55
    Hinv = torch.matmul(torch.matmul(cam.K, R.transpose(1, 2)), cam.K_inv)   # :56-57
    return H, R, Hinv


def _pick(v, ref, op):
    """op(v) where the elements attaining op are chosen on `ref`; ties share the gradient evenly, as torch's min / max do."""
    m = (ref == op(ref)) | (torch.isnan(ref) & torch.isnan(op(ref)))
    return (v * m).sum() / m.sum()


def frame_scale(cam, H, decide_H=None):
    """:125-143 -> dict of px_min, py_min, kw, kh, ikw, ikh, w_max, h_max, each (B,).  min / max reduce the 1-D tensor of one
    frame's four corners; the 4:3 branch is a Python `if` on the values.  decide_H: fp32 homographies whose corners choose
    the min / max corners and the branch instead (fp64 values with the fp32 forward's decisions, as vidc_frame_params_backward
    takes them)."""
    out = {k: [] for k in FIELDS[3:]}
    for i in range(H.shape[0]):
        c = torch.mm(H[i], cam.corners)                          # :125, one frame's (3,3) @ (3,4)
        px, py = c[0] / c[2], c[1] / c[2]                        # :126
        if decide_H is None:
            px_max, px_min = torch.max(px), torch.min(px)        # :127-130
            py_max, py_min = torch.max(py), torch.min(py)
            h_max, w_max = py_max - py_min, px_max - px_min      # :132-133
            wide = bool(w_max > (4 * h_max) / 3)                 # :135
        else:
            c32 = torch.mm(decide_H[i].float(), cam.corners.float())
            rx, ry = c32[0] / c32[2], c32[1] / c32[2]
            px_max, px_min = _pick(px, rx, torch.max), _pick(px, rx, torch.min)
            py_max, py_min = _pick(py, ry, torch.max), _pick(py, ry, torch.min)
            h_max, w_max = py_max - py_min, px_max - px_min
            wide = bool((rx.max() - rx.min()) > (4 * (ry.max() - ry.min())) / 3)
        if wide:
            kw = cam.W / w_max                                   # :136
            kh = cam.H / ((3 * w_max) / 4)                       # :137
        else:
            kh = cam.H / h_max                                   # :139
            kw = cam.W / ((4 * h_max) / 3)                       # :140
        for k, v in (("px_min", px_min), ("py_min", py_min), ("kw", kw), ("kh", kh), ("ikw", 1. / kw), ("ikh", 1. / kh),
                     ("w_max", w_max), ("h_max", h_max)):
            out[k].append(v)
    return {k: torch.stack(v) for k, v in out.items()}


def params(cam, I_g, I_a, decide_H=None):
    H, R, Hinv = build_homography(cam, I_g, I_a)
    p = frame_scale(cam, H, decide_H)
    p.update(H=H, R=R, Hinv=Hinv)
    return p


def _pixels(cam, dtype, device):
    Y, X = torch.meshgrid(torch.arange(cam.H, dtype=dtype, device=device), torch.arange(cam.W, dtype=dtype, device=device),
                          indexing="ij")
    return X.reshape(-1), Y.reshape(-1)


def forward_grid(cam, p):
    """:142-150 -> (B, H, W, 2) sampling grid of the forward warp."""
    X, Y = _pixels(cam, p["H"].dtype, p["H"].device)
    B = p["H"].shape[0]
    P = torch.stack([X * p["ikw"][:, None] + p["px_min"][:, None], Y * p["ikh"][:, None] + p["py_min"][:, None],
                     torch.ones(B, X.numel(), dtype=X.dtype, device=X.device)], 1)          # :142-145
    Q = torch.matmul(p["Hinv"], P)
    sx, sy = Q[:, 0] / Q[:, 2], Q[:, 1] / Q[:, 2]                          # :146-147
    gx, gy = cam.ihw * (sx - cam.cx), cam.ihh * (sy - cam.cy)              # :149-150
    return torch.stack([gx, gy], -1).reshape(B, cam.H, cam.W, 2)


def inverse_grid(cam, p):
    """:242-249 -> (B, H, W, 2) sampling grid of the inverse warp."""
    X, Y = _pixels(cam, p["H"].dtype, p["H"].device)
    B = p["H"].shape[0]
    P = torch.stack([X, Y, torch.ones_like(X)], 0).expand(B, 3, X.numel())
    Q = torch.matmul(p["H"], P)
    tx, ty = Q[:, 0] / Q[:, 2], Q[:, 1] / Q[:, 2]                          # :245
    cxp, cyp = p["kw"][:, None] * (tx - p["px_min"][:, None]), p["kh"][:, None] * (ty - p["py_min"][:, None])   # :246-247
    gx, gy = cam.ihw * (cxp - cam.cx), cam.ihh * (cyp - cam.cy)            # :248-249
    return torch.stack([gx, gy], -1).reshape(B, cam.H, cam.W, 2)


def warp(cam, x, I_g, I_a, mode="bilinear"):
    """warp_with_gravity_center_aligned (:108-156) -> (Cg_H_C, y)."""
    p = params(cam, I_g, I_a)
    y = F.grid_sample(x, forward_grid(cam, p).to(x.dtype), mode=mode, padding_mode="zeros", align_corners=False)   # :152
    return p["H"], y


def inverse_warp(cam, x, I_g, I_a):
    """inverse_warp_normal_image_with_gravity_center_aligned (:216-255) -> (Cg_H_C, z)."""
    p = params(cam, I_g, I_a)
    n = F.grid_sample(x, inverse_grid(cam, p).to(x.dtype), mode="bilinear", padding_mode="zeros", align_corners=False)   # :251
    B = x.shape[0]
    z = torch.bmm(p["R"].transpose(1, 2), n.reshape(B, 3, -1)).reshape(n.shape)                                        # :253
    return p["H"], z


def gravity_grads(fn, I_g, I_a, dtype):
    """(dL/dI_g, dL/dI_a) of the scalar fn(I_g, I_a) in `dtype`, from torch's autograd."""
    g = torch.tensor(np.asarray(I_g), dtype=dtype, requires_grad=True)
    a = torch.tensor(np.asarray(I_a), dtype=dtype, requires_grad=True)
    fn(g, a).backward()
    return g.grad.numpy().astype(np.float64), a.grad.numpy().astype(np.float64)
