"""normal_utils.py (DESIGN rows a9-a11) at its edges, on the CUDA path.

Losses: compute_normal_vectors_loss_l1 (both normalize_prediction settings) and compute_normal_vectors_loss_l2, through
the public functions and their autograd, against tests/loss_reference.py (the reference's expressions in plain torch,
differentiated by torch autograd on CPU) over its edge matrix: a norm sweep from 1e-45 to 1e30 with points at and one
ulp either side of both clamps (1e-12, 1e-8) and both overflow points (cube ~6.98e12, square ~1.84e19), signed zeros,
denormals, NaN and inf, degenerate geometry, every mask kind, pred layouts and upstream gradients.  One test per case
and mode, so a failure names its case.  Gradients use the term-scaled bar of loss_reference.grad_mismatches.

Helpers: Normalize, validity_mask, pyramid_masks and the C entry vidc_mask_nearest, bit for bit against the oracle or
torch on CPU.  Each helper input states which kernel it reaches; the dispatch conditions are those of
vidc_normalize3 / vidc_validity_mask (unit-stride contiguous planes, H*W % 4 == 0, frame stride % 4 == 0, 16-byte
aligned pointers -> *_vec4_kernel, anything else -> the generic kernel), and test_helpers_reach_the_intended_kernel
checks that claim with the profiler.
"""
import ctypes

import numpy as np
import pytest

from tests import common as C
from tests import loss_reference as LR

pytestmark = pytest.mark.gpu
CASES = LR.edge_cases()


def _fn(mode):
    from vi_depth_completion_b200 import normal_utils as NU
    if mode == "l1":
        return lambda p, g, m: NU.compute_normal_vectors_loss_l1(g, p, m)
    if mode == "l1_raw":
        return lambda p, g, m: NU.compute_normal_vectors_loss_l1(g, p, m, normalize_prediction=False)
    return lambda p, g, m: NU.compute_normal_vectors_loss_l2(g, p, m)


def _leaf(pred, layout, dev):
    """(leaf with requires_grad, the pred view handed to the loss, function reading pred's gradient from the leaf)."""
    import torch
    x = torch.from_numpy(pred).to(dev)
    if layout == "channels_last":
        leaf = x.contiguous(memory_format=torch.channels_last).requires_grad_(True)
        return leaf, leaf, lambda: leaf.grad
    if layout == "strided":               # a slice of a wider tensor: channel, row and column strides all non-trivial
        B, Cc, H, W = x.shape
        wide = torch.zeros(B, Cc + 3, H, W + 5, device=dev)
        wide[:, 2:2 + Cc, :, 3:3 + W] = x
        wide.requires_grad_(True)
        view = wide[:, 2:2 + Cc, :, 3:3 + W]
        assert not view.is_contiguous()
        return wide, view, lambda: wide.grad[:, 2:2 + Cc, :, 3:3 + W]
    leaf = x.clone().requires_grad_(True)
    return leaf, leaf, lambda: leaf.grad


def _scalar_ok(ours, ref, scale, rel=2e-5):
    ours, ref = float(ours), float(ref)
    if np.isnan(ref) or np.isnan(ours):
        return np.isnan(ref) and np.isnan(ours)
    if np.isinf(ref) or np.isinf(ours):
        return ours == ref
    return abs(ours - ref) <= rel * scale + 1e-30


def _loss_scales(mode, case):
    """Scale of the l2 loss (fp64): the magnitudes of the terms of every cosine, sum_c |r_c g_c| / (N1 N2), summed over
    pixels and divided by |sum(mask)| (a cosine of pred perpendicular to gt is pure cancellation residue).  None for the
    L1 losses and the angle, whose terms are absolute values and non-negative angles: |value| is their scale."""
    if mode != "l2":
        return None
    r = case["pred"][:, 0:3].astype(np.float64)
    g = case["gt"].astype(np.float64)
    m = LR.as_mask4(case["mask"]).numpy().astype(np.float64)
    with np.errstate(all="ignore"):
        n1 = np.maximum(np.sqrt((r * r).sum(1)), 1e-8)
        n2 = np.maximum(np.sqrt((g * g).sum(1)), 1e-8)
        return float(np.sum(np.abs(r * g).sum(1) / (n1 * n2)) / np.abs(m.sum()))


@pytest.mark.parametrize("mode", LR.MODES)
@pytest.mark.parametrize("name", sorted(CASES))
def test_loss_and_gradient_match_torch_on_edges(cuda_device, name, mode):
    import torch
    case = CASES[name]
    leaf, p, grad_of = _leaf(case["pred"], case["layout"], cuda_device)
    gt = torch.from_numpy(case["gt"]).to(cuda_device)
    mask = torch.from_numpy(np.ascontiguousarray(case["mask"])).to(cuda_device)
    loss, angle = _fn(mode)(p, gt, mask)
    outer = LR.outer_fn(case)
    (outer(loss) if outer is not None else loss * float(case["up"])).backward()
    rloss, rangle, rgrad = LR.reference(mode, case["pred"], case["gt"], case["mask"], case["up"], outer)

    l2_scale = _loss_scales(mode, case)
    lscale = l2_scale if l2_scale is not None else abs(float(rloss))
    assert _scalar_ok(loss.detach().cpu(), rloss, lscale), f"{name}/{mode}: loss {float(loss)} vs torch {rloss}"
    assert _scalar_ok(angle.cpu(), rangle, abs(float(rangle))), f"{name}/{mode}: angle {float(angle)} vs torch {rangle}"

    d = grad_of().detach().cpu().numpy()
    m = LR.as_mask4(case["mask"]).numpy()
    with np.errstate(all="ignore"):
        go = np.float32(LR.effective_up(case)) / np.float32(np.sum(m, dtype=np.float64))
    bad = LR.grad_mismatches(mode, d, rgrad, case["pred"], case["gt"], case["mask"], go)
    if bad.any():
        idx = np.argwhere(bad)[:4]
        where = "; ".join(f"(b={b}, c={c}, y={y}, x={x}) pred={case['pred'][b, :3, y, x]} cuda={d[b, c, y, x]:.6g} "
                          f"torch={rgrad[b, c, y, x]:.6g}" for b, c, y, x in idx)
        pytest.fail(f"{name}/{mode}: {int(bad.sum())} gradient components off: {where}")
    assert np.array_equal(d[:, 3:], np.zeros_like(d[:, 3:])), f"{name}/{mode}: channels >= 3 must get exact zeros"
    if case["layout"] == "strided":
        full = leaf.grad.clone()
        full[:, 2:2 + case["pred"].shape[1], :, 3:3 + case["pred"].shape[3]] = 0
        assert torch.count_nonzero(full).item() == 0, "the gradient reached elements outside the view"


def test_large_reduction_is_exact(cuda_device):
    """64 x 480 x 640 pixels: sum(mask) of a 0/1 mask must be the exact count (the loss divides by it), the angle sum
    within 1e-6 of an fp64 sum of torch's per-pixel angles, and both losses within 1e-6 of fp64 sums of torch's terms."""
    import torch
    import torch.nn.functional as F
    from vi_depth_completion_b200 import normal_utils as NU
    B, H, W = 64, 480, 640
    gen = torch.Generator().manual_seed(123)
    pred = torch.randn(B, 3, H, W, generator=gen)
    gt = F.normalize(torch.randn(B, 3, H, W, generator=gen), dim=1)
    mask = (torch.rand(B, 1, H, W, generator=gen) < 0.6).float()
    count = int(mask.sum(dtype=torch.float64).item())
    dp, dg, dm = pred.to(cuda_device), gt.to(cuda_device), mask.to(cuda_device)
    s = NU._stats(dg, dp, dm, True).cpu().numpy()
    assert s[1] == count, f"sum(mask) = {s[1]!r}, the mask has {count} ones"
    n = F.normalize(pred, dim=1)
    ang = (torch.acos(torch.clamp(torch.sum(n * gt, 1, keepdim=True), -1, 1)) / np.pi * 180 * mask).double().sum().item()
    l1_terms = (n * mask - gt * mask).abs().double().sum().item()
    cos = F.cosine_similarity(pred, gt, dim=1).double()
    del n
    loss1, angle = NU.compute_normal_vectors_loss_l1(dg, dp, dm)
    loss2, _ = NU.compute_normal_vectors_loss_l2(dg, dp, dm)
    assert abs(float(angle) - ang) <= 1e-6 * ang
    assert abs(float(loss1) - l1_terms / count) <= 1e-6 * l1_terms / count
    assert abs(float(loss2) + cos.sum().item() / count) <= 1e-6 * cos.abs().sum().item() / count


# ---- Normalize (vidc_normalize3) ---------------------------------------------------------------------------------------------
def _normalize_into(x, out):
    """vidc_normalize3 through the C ABI, into a caller-provided output view."""
    import torch
    from vi_depth_completion_b200._cabi import check, lib
    from vi_depth_completion_b200.warping_2dof_alignment import _image, _stream_ptr
    xi, oi = _image(x), _image(out)
    with torch.cuda.device(x.device):
        check(lib().vidc_normalize3(ctypes.byref(xi), ctypes.byref(oi), _stream_ptr(x.device)))
    return out


def _normalize_inputs():
    _, _, sv = C.special_value_images(3, 30, 24, seed=5)           # H*W = 720, a multiple of 4
    _, _, odd = C.special_value_images(3, 31, 23, seed=6)          # H*W = 713
    return sv.astype(np.float32), odd.astype(np.float32)


def _run_normalize(path, dev):
    """(result, oracle input) of one Normalize call; `path` names the input and, by it, the kernel it reaches."""
    import torch
    from vi_depth_completion_b200 import normal_utils as NU
    sv, odd = _normalize_inputs()
    if path == "vec4_contiguous":                      # contiguous planes, H*W % 4 == 0, aligned: normalize3_vec4_kernel
        return NU.Normalize(torch.from_numpy(sv).to(dev)), sv
    if path == "generic_hw_not_multiple_of_4":         # H*W % 4 != 0: normalize3_kernel
        return NU.Normalize(torch.from_numpy(odd).to(dev)), odd
    if path == "generic_channels_last":                # channel stride 1 (input and the empty_like output): normalize3_kernel
        return NU.Normalize(torch.from_numpy(sv).to(dev).contiguous(memory_format=torch.channels_last)), sv
    if path == "generic_strided_view":                 # row stride != W: normalize3_kernel
        wide = torch.full((3, 5, 30, 24 + 7), float("nan"), device=dev)
        wide[:, 1:4, :, 2:26] = torch.from_numpy(sv).to(dev)
        return NU.Normalize(wide[:, 1:4, :, 2:26]), sv
    if path == "generic_output_4_bytes_in":            # output pointer 4 bytes past a 16-byte boundary: normalize3_kernel
        buf = torch.full((sv.size + 1,), float("nan"), device=dev)
        out = buf[1:].view(sv.shape)
        assert out.data_ptr() % 16 == 4
        _normalize_into(torch.from_numpy(sv).to(dev), out)
        assert torch.isnan(buf[0]).item(), "normalize3 wrote before its output"
        return out, sv
    raise AssertionError(path)


NORMALIZE_PATHS = ["vec4_contiguous", "generic_hw_not_multiple_of_4", "generic_channels_last", "generic_strided_view",
                   "generic_output_4_bytes_in"]


@pytest.mark.parametrize("path", NORMALIZE_PATHS)
def test_normalize_matches_oracle_bits(cuda_device, oracle_mod, path):
    """F.normalize(dim=1) on the special-value images (signed zeros, denormals, huge values, inf, NaN)."""
    out, x = _run_normalize(path, cuda_device)
    with np.errstate(all="ignore"):
        want = oracle_mod.normalize(x)
    assert C.count_bit_mismatches(out.cpu().numpy(), want) == 0


# ---- validity_mask (vidc_validity_mask) --------------------------------------------------------------------------------------
def _mask_input(H, W, Cc, seed):
    """(B=3, Cc, H, W): frame 0 holds the threshold edges (sums exactly 0.01f and one ulp either side, reached through
    one component and through a three-term sum), -0, NaN and +inf + -inf; frames 1-2 are values near the threshold."""
    rs = np.random.RandomState(seed)
    x = (rs.rand(3, Cc, H, W).astype(np.float32) * np.float32(0.02 / 3)).astype(np.float32)
    t = np.float32(0.01)
    lo, hi = np.nextafter(t, np.float32(0)), np.nextafter(t, np.float32(1))
    edges = [(t, 0, 0), (lo, 0, 0), (hi, 0, 0), (0, t, 0), (0, 0, hi), (-0.0, -0.0, -0.0), (0.0, -0.0, 0.0),
             (np.nan, 1, 1), (1, np.nan, 0), (np.inf, -np.inf, 1), (np.inf, 0, -np.inf), (np.inf, 0, 0),
             (-np.inf, 1, 1), (0.005, 0.005, 0.0), (np.float32(0.01 / 3),) * 3, (hi, -0.0, 0.0), (1e-45, t, 0)]
    flat = x[0, :3].reshape(3, -1)
    for i, e in enumerate(edges):
        flat[:, 7 * i % flat.shape[1]] = np.array(e, np.float32)
    x[0, :3] = flat.reshape(3, H, W)
    return x


def _mask_reference(x):
    import torch
    t = torch.from_numpy(x)
    return (t[:, 0:1] + t[:, 1:2] + t[:, 2:3] > 1e-2).float().numpy()


MASK_PATHS = ["vec4_contiguous", "vec4_four_channels", "generic_hw_not_multiple_of_4", "generic_channels_last",
              "generic_strided_view"]


def _mask_tensor(path, dev):
    import torch
    if path == "vec4_contiguous":                      # validity_mask_vec4_kernel
        x = _mask_input(24, 20, 3, 1)
        return torch.from_numpy(x).to(dev), x
    if path == "vec4_four_channels":                   # C = 4, still contiguous planes: validity_mask_vec4_kernel
        x = _mask_input(24, 20, 4, 2)
        return torch.from_numpy(x).to(dev), x
    if path == "generic_hw_not_multiple_of_4":         # H*W = 21*19: validity_mask_kernel
        x = _mask_input(21, 19, 3, 3)
        return torch.from_numpy(x).to(dev), x
    if path == "generic_channels_last":                # validity_mask_kernel
        x = _mask_input(24, 20, 4, 4)
        return torch.from_numpy(x).to(dev).contiguous(memory_format=torch.channels_last), x
    if path == "generic_strided_view":                 # row stride != W: validity_mask_kernel
        x = _mask_input(24, 20, 3, 5)
        wide = torch.full((3, 4, 24, 29), float("nan"), device=dev)
        wide[:, :3, :, 4:24] = torch.from_numpy(x).to(dev)
        return wide[:, :3, :, 4:24], x
    raise AssertionError(path)


@pytest.mark.parametrize("as_float", [True, False], ids=["float", "uint8"])
@pytest.mark.parametrize("path", MASK_PATHS)
def test_validity_mask_matches_torch(cuda_device, path, as_float):
    import torch
    from vi_depth_completion_b200 import normal_utils as NU
    x_dev, x = _mask_tensor(path, cuda_device)
    want = _mask_reference(x)
    m = NU.validity_mask(x_dev, as_float=as_float)
    assert m.dtype == (torch.float32 if as_float else torch.uint8) and tuple(m.shape) == want.shape
    assert np.array_equal(m.cpu().numpy().astype(np.float32), want)
    m2, cov = NU.validity_mask(x_dev, as_float=as_float, with_coverage=True)
    assert torch.equal(m2, m)
    assert cov.dtype == torch.int32
    assert cov.cpu().numpy().tolist() == want.reshape(want.shape[0], -1).sum(1).astype(np.int64).tolist()


# ---- pyramid_masks (vidc_mask_pyramid) and vidc_mask_nearest ------------------------------------------------------------------
def _size_pairs(seed, n):
    """(Hin, Win, Hout, Wout) with down- and up-sampling, 489-row inputs, 1x1 outputs, identity and exact 2x."""
    rs = np.random.RandomState(seed)
    pairs = [(489, 640, 60, 80), (489, 640, 1, 1), (480, 640, 8, 10), (1, 1, 7, 5), (7, 9, 14, 18), (13, 17, 13, 17),
             (489, 3, 490, 2), (5, 489, 1, 977), (240, 320, 60, 80), (2, 2, 1, 1)]
    for _ in range(n):
        hin, win = int(rs.randint(1, 500)), int(rs.randint(1, 500))
        pairs.append((hin, win, int(rs.randint(1, 2 * hin + 2)), int(rs.randint(1, 2 * win + 2))))
    return pairs


def _nearest(m, h, w):
    import torch
    return torch.nn.functional.interpolate(torch.from_numpy(m), size=(h, w), mode="nearest").numpy()


@pytest.mark.parametrize("source", ["float_binary", "float_nonbinary", "uint8"])
def test_pyramid_masks_match_interpolate(cuda_device, source):
    import torch
    from vi_depth_completion_b200 import normal_utils as NU
    rs = np.random.RandomState({"float_binary": 1, "float_nonbinary": 2, "uint8": 3}[source])
    pairs = _size_pairs(10 + len(source), 24)
    i = 0
    while i < len(pairs):
        hin, win = pairs[i][:2]
        levels = int(rs.randint(1, 5))
        sizes = [(p[2], p[3]) for p in pairs[i:i + levels]]
        i += levels
        B = 2
        if source == "float_nonbinary":
            m = np.array([0.0, 0.3, 1.0, 2.5, -1.0, -0.0], np.float32)[rs.randint(0, 6, size=(B, 1, hin, win))]
        else:
            m = (rs.rand(B, 1, hin, win) < 0.5).astype(np.float32)
        src = torch.from_numpy(m.astype(np.uint8) if source == "uint8" else m).to(cuda_device)
        outs = NU.pyramid_masks(src, sizes)
        assert len(outs) == len(sizes)
        for (h, w), o in zip(sizes, outs):
            got = o.cpu().numpy()
            assert C.count_bit_mismatches(got, _nearest(m, h, w)) == 0, f"{source}: {hin}x{win} -> {h}x{w}"


def test_pyramid_masks_default_sizes_cover_every_level_count(cuda_device):
    import torch
    from vi_depth_completion_b200 import normal_utils as NU
    m = (np.random.RandomState(4).rand(3, 1, 489, 640) < 0.5).astype(np.float32)
    for levels in range(1, 5):
        sizes = NU.PYRAMID_SIZES[:levels]
        outs = NU.pyramid_masks(torch.from_numpy(m).to(cuda_device), sizes)
        for (h, w), o in zip(sizes, outs):
            assert np.array_equal(o.cpu().numpy(), _nearest(m, h, w))


def test_mask_nearest_c_entry_matches_interpolate(cuda_device):
    import torch
    from vi_depth_completion_b200._cabi import check, lib
    from vi_depth_completion_b200.warping_2dof_alignment import _stream_ptr
    rs = np.random.RandomState(7)
    for hin, win, hout, wout in _size_pairs(8, 40):
        m = np.array([0.0, 1.0, 0.5, -2.0], np.float32)[rs.randint(0, 4, size=(2, 1, hin, win))]
        src = torch.from_numpy(m).to(cuda_device)
        out = torch.full((2, 1, hout, wout), float("nan"), device=cuda_device)
        with torch.cuda.device(cuda_device):
            check(lib().vidc_mask_nearest(src.data_ptr(), 2, hin, win, hout, wout, out.data_ptr(), _stream_ptr(cuda_device)))
        assert C.count_bit_mismatches(out.cpu().numpy(), _nearest(m, hout, wout)) == 0, f"{hin}x{win} -> {hout}x{wout}"


# ---- which kernel each helper input reaches ----------------------------------------------------------------------------------
def _kernel_names(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " | ".join(sorted({e.name for e in prof.events()}))


def test_helpers_reach_the_intended_kernel(cuda_device):
    """The path names used above are true: the generic kernels are exercised, not only the vec4 ones."""
    from vi_depth_completion_b200 import normal_utils as NU
    for path in NORMALIZE_PATHS:
        names = _kernel_names(lambda: _run_normalize(path, cuda_device))
        want = "normalize3_vec4_kernel" if path.startswith("vec4") else "normalize3_kernel"
        other = "normalize3_kernel" if path.startswith("vec4") else "normalize3_vec4_kernel"
        assert want in names and other not in names, f"{path}: {names}"
    for path in MASK_PATHS:
        x_dev, _ = _mask_tensor(path, cuda_device)
        names = _kernel_names(lambda: NU.validity_mask(x_dev, with_coverage=True))
        want = "validity_mask_vec4_kernel" if path.startswith("vec4") else "validity_mask_kernel"
        other = "validity_mask_kernel" if path.startswith("vec4") else "validity_mask_vec4_kernel"
        assert want in names and other not in names, f"{path}: {names}"
