"""Plain-torch restatement of the two losses of normal_utils.py (:7-34) and a numpy fp32 model of
normal_loss_backward_kernel (csrc/kernels_generic.cuh), for tests.

`reference` evaluates the losses exactly as the reference writes them (Normalize := F.normalize(dim=1)) on CPU tensors
and differentiates them with torch autograd; it reproduces tests/golden/golden_tiny_loss_backward.npz, which was frozen
from the executed reference.  `grad_tolerance` gives each gradient component a bar that scales with the magnitudes of
the terms summed into it (fp64), so cancellation residue is not mistaken for an error.  `kernel_model` restates the CUDA
backward op for op in fp32 (the library is built with -fmad=false), so a divergence between the kernel's arithmetic and
torch's chain rule shows on any machine.
"""
import numpy as np
import torch
import torch.nn.functional as F

from tests.common import special_value_images

MODES = ("l1", "l1_raw", "l2")
REL = 2e-5


def _l1(p, gt, m, normalize=True):                       # normal_utils.py:20-34
    n = F.normalize(p[:, 0:3], dim=1) if normalize else p[:, 0:3]
    angle = torch.sum(torch.acos(torch.clamp(torch.sum(n * gt, 1, keepdim=True), -1, 1)) / np.pi * 180 * m)
    return torch.nn.L1Loss(reduction='sum')(n * m, gt * m) / torch.sum(m).item(), angle


def _l2(p, gt, m):                                        # normal_utils.py:7-17 (the cosine term is NOT masked)
    n = F.normalize(p[:, 0:3], dim=1)
    angle = torch.sum(torch.acos(torch.clamp(torch.sum(n * gt, 1, keepdim=True), -1, 1)) / np.pi * 180 * m)
    return -torch.sum(F.cosine_similarity(p[:, 0:3], gt, dim=1)) / torch.sum(m).item(), angle


def as_mask4(mask):
    """The mask as the losses see it: float, (B,1,H,W) (normal_utils.py:21; a (B,H,W) mask gets its channel axis)."""
    m = torch.as_tensor(mask).float()
    return m.unsqueeze(1) if m.dim() == 3 else m


def reference(mode, pred, gt, mask, up=1.0, outer=None):
    """(loss, angle, grad) of `mode` on CPU: loss and angle as float32 scalars, grad = d(outer(loss)) / d pred as float32
    (B,C,H,W).  outer defaults to loss * up; pass another function to use the loss more than once in one graph."""
    p = torch.as_tensor(np.asarray(pred, np.float32)).clone().requires_grad_(True)
    g = torch.as_tensor(np.asarray(gt, np.float32))
    m = as_mask4(mask)
    if mode == "l2":
        loss, angle = _l2(p, g, m)
    else:
        loss, angle = _l1(p, g, m, normalize=(mode == "l1"))
    total = outer(loss) if outer is not None else loss * float(up)
    total.backward()
    return np.float32(loss.detach().item()), np.float32(angle.detach().item()), p.grad.numpy().copy()


def grad_tolerance(mode, pred, gt, mask, go):
    """Per-component scale (B,3,H,W) of the backward: the magnitudes of the terms summed into each component, in fp64.
    go = upstream gradient / sum(mask).  l1: |dn_c / N| + |k r_c|; l2: |go g_c / (N1 N2)| + |go k r_c|; l1_raw: |dn_c|,
    with dn_c = go m (the sign factor taken as 1) and k built from the absolute values of the terms of its dot product.
    Non-finite scales are returned as inf (the comparison then falls back to the reference's own magnitude)."""
    r = np.asarray(pred, np.float64)[:, 0:3]
    g = np.asarray(gt, np.float64)
    m = as_mask4(mask).numpy().astype(np.float64)
    go = abs(float(go))
    with np.errstate(all="ignore"):
        nr = np.sqrt((r * r).sum(1, keepdims=True))
        if mode == "l1_raw":
            s = np.broadcast_to(go * np.abs(m), r.shape).copy()
        elif mode == "l1":
            N = np.maximum(nr, 1e-12)
            dn = go * np.abs(m)
            k = np.where(nr >= 1e-12, (dn * np.abs(r)).sum(1, keepdims=True) / (N * N * nr), 0.0)
            s = dn / N + k * np.abs(r)
        else:
            N1 = np.maximum(nr, 1e-8)
            N2 = np.maximum(np.sqrt((g * g).sum(1, keepdims=True)), 1e-8)
            k = np.where(nr > 0, (np.abs(g) * np.abs(r)).sum(1, keepdims=True) / (N2 * N1 * N1 * nr), 0.0)
            s = go * np.abs(g) / (N1 * N2) + go * k * np.abs(r)
    return np.where(np.isfinite(s), s, np.inf)


def grad_mismatches(mode, d, ref, pred, gt, mask, go, rel=REL):
    """Boolean (B,3,H,W) of gradient components that miss the reference: NaN where the reference is not NaN (or the
    reverse), an infinity of another sign, or a finite error above rel * term scale.  Where the term scale is not finite
    the bar is rel * |ref|.  Zeros of either sign are equal."""
    d = np.asarray(d, np.float64)[:, 0:3]
    ref = np.asarray(ref, np.float64)[:, 0:3]
    scale = grad_tolerance(mode, pred, gt, mask, go)
    scale = np.where(np.isfinite(scale), scale, np.abs(ref))
    nan_d, nan_r = np.isnan(d), np.isnan(ref)
    inf_r = np.isinf(ref)
    with np.errstate(all="ignore"):
        err = np.abs(d - ref)
    bad = nan_d != nan_r
    bad |= inf_r & ~nan_d & (d != ref)
    fin = ~nan_r & ~inf_r
    bad |= fin & ~nan_d & ~(err <= rel * scale)
    return bad


def _nan_keeping_clamp_min(x, lo):
    return np.where(x < lo, np.float32(lo), x).astype(np.float32)


def kernel_model(mode, pred, gt, mask, up=1.0, sum_mask=None):
    """normal_loss_backward_kernel restated op for op in numpy fp32 (no fused multiply-add), returning (B,C,H,W)."""
    f = np.float32
    r = [np.asarray(pred, f)[:, c] for c in range(3)]
    g = [np.asarray(gt, f)[:, c] for c in range(3)]
    m = as_mask4(mask).numpy()[:, 0]
    if sum_mask is None:
        sum_mask = float(np.sum(m, dtype=np.float64))
    zero = f(0.0)
    with np.errstate(all="ignore"):
        go = f(up) / f(sum_mask)
        nr = np.sqrt((r[0] * r[0] + r[1] * r[1]) + r[2] * r[2])
        if mode == "l2":
            ng = np.sqrt((g[0] * g[0] + g[1] * g[1]) + g[2] * g[2])
            n1 = _nan_keeping_clamp_min(nr, f(1e-8))
            n2 = _nan_keeping_clamp_min(ng, f(1e-8))
            ga = [-go * (g[c] / n2) for c in range(3)]
            dd = [ga[c] * ((r[c] / n1) / n1) for c in range(3)]
            gn = -((dd[0] + dd[1]) + dd[2])
            d = [ga[c] / n1 + gn * np.where(nr == 0, zero, r[c] / nr) for c in range(3)]
        else:
            nn = _nan_keeping_clamp_min(nr, f(1e-12))
            n = [r[c] / nn for c in range(3)] if mode == "l1" else r
            dn = []
            for c in range(3):
                diff = n[c] * m - g[c] * m
                sg = np.where(diff > 0, f(1.0), np.where(diff < 0, f(-1.0), zero))
                dn.append(go * sg * m)
            if mode == "l1":
                dd = [dn[c] * ((r[c] / nn) / nn) for c in range(3)]
                gn = np.where(nr >= f(1e-12), -((dd[0] + dd[1]) + dd[2]), zero)
                d = [dn[c] / nn + gn * np.where(nr == 0, zero, r[c] / nr) for c in range(3)]
            else:
                d = dn
    out = np.zeros(np.asarray(pred).shape, f)
    for c in range(3):
        out[:, c] = d[c]
    return out


# ---- edge matrix shared by the CPU check of kernel_model and the GPU check of the CUDA path --------------------------------
F32_MAX = np.finfo(np.float32).max
THRESHOLDS = {                                                   # norms where the chain rule changes form or overflows
    "normalize_clamp": np.float32(1e-12),                       # F.normalize: norm.clamp_min(1e-12)
    "cosine_clamp": np.float32(1e-8),                           # cosine_similarity: each norm clamp_min_(1e-8)
    "cube_overflow": np.float32(np.cbrt(np.float64(F32_MAX))),  # ~6.98e12: N^3 overflows in fp32
    "square_overflow": np.float32(np.sqrt(np.float64(F32_MAX))),  # ~1.84e19: the norm's own sum of squares overflows
}
GENERAL_DIR = np.array([3.0, -2.0, 5.0], np.float64) / np.sqrt(38.0)


def _unit(rs, n):
    v = rs.randn(n, 3)
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(np.float32)


def _pixels(r, g, m=None, W=16, C=4):
    """N per-pixel vectors -> one (1,C,H,W) frame (row-major), padded with benign pixels; channel 3+ is noise."""
    r = np.asarray(r, np.float32); g = np.asarray(g, np.float32)
    n = r.shape[0]
    H = -(-n // W)
    rs = np.random.RandomState(n)
    pad = H * W - n
    rp = np.concatenate([r, rs.randn(pad, 3).astype(np.float32)]) if pad else r
    gp = np.concatenate([g, _unit(rs, pad)]) if pad else g
    mp = np.ones(H * W, np.float32) if m is None else np.concatenate([np.asarray(m, np.float32), np.ones(pad, np.float32)])
    pred = np.empty((1, C, H, W), np.float32)
    pred[0, :3] = rp.T.reshape(3, H, W)
    if C > 3:
        pred[0, 3:] = rs.randn(C - 3, H, W)
    return pred, gp.T.reshape(1, 3, H, W).copy(), mp.reshape(1, 1, H, W)


def _directions(rs):
    """Axis-aligned vectors of both signs (their norm is exactly the scale) and two general directions."""
    e = np.eye(3)
    return np.concatenate([e, -e, GENERAL_DIR[None], _unit(rs, 1).astype(np.float64)])


def _scaled(scales, rs):
    d = _directions(rs)
    s = np.asarray(scales, np.float64)
    with np.errstate(over="ignore"):
        r = (s[:, None, None] * d[None]).reshape(-1, 3).astype(np.float32)
    return r


def _norm_case(scales, seed):
    rs = np.random.RandomState(seed)
    r = _scaled(scales, rs)
    return _pixels(r, _unit(rs, r.shape[0]))


def _threshold_case(t, seed):
    t = np.float32(t)
    pts = [np.nextafter(t, np.float32(0)), t, np.nextafter(t, np.float32(np.inf))]
    band = (np.float64(t) * np.logspace(-2, 2, 41)).astype(np.float32)
    return _norm_case(np.concatenate([pts, band]).astype(np.float32), seed)


def _special_components(vals, seed, all_three=False):
    rs = np.random.RandomState(seed)
    rows = []
    for v in vals:
        if all_three:
            rows += [[v, v, v], [v, -v, v]]
        else:
            for c in range(3):
                x = rs.randn(3).astype(np.float32)
                x[c] = v
                rows.append(x)
                y = np.zeros(3, np.float32)
                y[c] = v
                rows.append(y)
    r = np.array(rows, np.float32)
    return _pixels(r, _unit(rs, r.shape[0]))


def _random(B, H, W, seed, C=4):
    rs = np.random.RandomState(seed)
    pred = rs.randn(B, C, H, W).astype(np.float32)
    g = _unit(rs, B * H * W).reshape(B, H, W, 3).transpose(0, 3, 1, 2).copy()
    m = (rs.rand(B, 1, H, W) < 0.6).astype(np.float32)
    return pred, g, m


def _geometry(kind, seed):
    rs = np.random.RandomState(seed)
    g = _unit(rs, 96)
    s = np.array([1e-10, 1e-3, 0.5, 1.0, 3.0, 1e3, 1e10, 1e15], np.float32)
    s = np.tile(s, 12)
    if kind == "parallel":
        r = g * s[:, None]
    elif kind == "antiparallel":
        r = -g * s[:, None]
    else:
        r = np.cross(g, rs.randn(96, 3)).astype(np.float32)
        r = r / np.linalg.norm(r, axis=1, keepdims=True) * s[:, None]
    return _pixels(r.astype(np.float32), g)


def _gt_scaled(seed):
    rs = np.random.RandomState(seed)
    pred, g, m = _random(2, 8, 12, seed)
    sc = np.array([0.0, 1e-12, 1e-9, 1e-8, 1e-5, 0.3, 7.0, 1e5, 1e19], np.float32)
    f = sc[rs.randint(0, sc.size, size=(2, 1, 8, 12))]
    return pred, (g * f).astype(np.float32), m


def _special_images(seed):
    _, _, normals = special_value_images(3, 30, 20, seed)
    rs = np.random.RandomState(seed)
    g = _unit(rs, 3 * 30 * 20).reshape(3, 30, 20, 3).transpose(0, 3, 1, 2).copy()
    m = (rs.rand(3, 1, 30, 20) < 0.7).astype(np.float32)
    return normals.astype(np.float32), g, m


def _soft_mask(seed):
    rs = np.random.RandomState(seed)
    pred, g, _ = _random(2, 9, 13, seed)
    m = np.array([0.0, 0.25, 1.0, 2.0], np.float32)[rs.randint(0, 4, size=(2, 1, 9, 13))]
    return pred, g, m


def _zero_frame_mask(seed):
    pred, g, m = _random(3, 8, 10, seed)
    m[1] = 0
    return pred, g, m


def _zero_mask(seed):
    pred, g, m = _random(2, 6, 7, seed)
    return pred, g, np.zeros_like(m)


def _exact_match(seed):
    """pred == gt (l1_raw: diff exactly 0, sign(0) = 0) and pred == gt scaled (l1: normalised diff exactly 0 or 1 ulp)."""
    rs = np.random.RandomState(seed)
    g = _unit(rs, 64)
    g[:8] = np.eye(3, dtype=np.float32)[rs.randint(0, 3, 8)]
    return _pixels(g.copy(), g)


def edge_cases():
    """name -> dict(pred, gt, mask, up, outer, layout).  up is the upstream gradient of the scalar loss; outer, when not
    None, is a tuple of multipliers c_i of a graph sum_i loss * c_i that uses the loss more than once; layout names a
    memory layout the GPU test applies to pred (the arithmetic is layout-independent)."""
    cases = {}

    def add(name, arrays, up=1.7, outer=None, layout=None, mask_kind=None):
        pred, gt, m = arrays
        if mask_kind == "bool":
            m = m > 0
        elif mask_kind == "uint8":
            m = (m > 0).astype(np.uint8)
        elif mask_kind == "3d":
            m = m[:, 0]
        cases[name] = dict(pred=pred, gt=gt, mask=m, up=up, outer=outer, layout=layout)

    add("norm_sweep_1e-45_to_1e30", _norm_case(np.logspace(-45, 30, 301).astype(np.float32), 1))
    for i, (tname, t) in enumerate(THRESHOLDS.items()):
        add(f"norm_at_{tname}", _threshold_case(t, 10 + i))
    add("zero_vectors_signed", _pixels(np.array([[a, b, c] for a in (0.0, -0.0) for b in (0.0, -0.0) for c in (0.0, -0.0)],
                                                np.float32), _unit(np.random.RandomState(3), 8)))
    add("denormal_single_component", _special_components([1e-45, -1e-45, 1e-40, -3e-39, 1.1754942e-38], 4))
    add("nan_one_component", _special_components([np.nan], 5))
    add("nan_all_components", _special_components([np.nan], 6, all_three=True))
    add("inf_one_component", _special_components([np.inf, -np.inf], 7))
    add("inf_all_components", _special_components([np.inf, -np.inf], 8, all_three=True))
    add("special_value_images", _special_images(21))
    for i, kind in enumerate(("parallel", "antiparallel", "perpendicular")):
        add(f"pred_{kind}_to_gt", _geometry(kind, 30 + i))
    add("pred_equals_gt", _exact_match(33))
    pred, g, m = _random(2, 7, 9, 34)
    add("gt_zero", (pred, np.zeros_like(g), m))
    add("gt_scaled", _gt_scaled(35))
    add("mask_soft_values", _soft_mask(36))
    add("mask_bool", _random(2, 7, 11, 37), mask_kind="bool")
    add("mask_uint8", _random(2, 7, 11, 38), mask_kind="uint8")
    add("mask_3d", _random(2, 7, 11, 39), mask_kind="3d")
    add("mask_zero_in_one_frame", _zero_frame_mask(40))
    add("mask_zero_everywhere", _zero_mask(41))
    add("pred_3_channels", _random(2, 8, 8, 42, C=3))
    add("pred_7_channels", _random(2, 8, 8, 43, C=7))
    add("pred_channels_last", _random(2, 9, 10, 44), layout="channels_last")
    add("pred_strided_view", _random(2, 9, 10, 45), layout="strided")
    add("odd_size_37x11", _random(2, 37, 11, 46))
    add("odd_size_9x70", _random(1, 9, 70, 47))
    add("batch_1", _random(1, 16, 40, 48))
    add("batch_300", _random(300, 5, 6, 49))
    add("upstream_zero", _random(2, 6, 9, 50), up=0.0)
    add("upstream_negative", _random(2, 6, 9, 51), up=-2.5)
    add("loss_used_twice", _random(2, 6, 9, 52), outer=(1.5, -0.25))
    return cases


def outer_fn(case):
    if case["outer"] is None:
        return None
    cs = case["outer"]
    return lambda loss: sum(loss * c for c in cs)


def effective_up(case):
    """The gradient that reaches the loss node: the multipliers of every use, summed in fp32 by autograd."""
    if case["outer"] is None:
        return np.float32(case["up"])
    acc = np.float32(0.0)
    for c in case["outer"]:
        acc = np.float32(acc + np.float32(c))
    return acc
