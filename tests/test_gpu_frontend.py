"""The thin torch C++ extension (csrc/torch_ops.cpp, `torch.ops.vidc.*`) in front of the C ABI: the only route of the hot
entry points, reference error behaviour, traceable by torch.compile(fullgraph=True)."""
import numpy as np
import pytest

from tests import common as C

pytestmark = pytest.mark.gpu


def _setup(dev, cam="S1", B=4):
    import torch
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    w = Warping2DOFAlignment(*C.CAMERAS[cam])
    H, W = int(w.H), int(w.W)
    I_g, I_a = C.random_gravity(B, seed=3)
    rgb, depth, normals = C.random_images(B, H, W, seed=2, sparse_depth=True)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    return w, t(rgb), t(depth), t(normals), t(I_g), t(I_a)


def test_extension_is_loaded_and_keeps_the_memory_format(cuda_device):
    """The hot entry points run through the loaded extension; channels-last input gives channels-last output.  Their bits
    against the oracle and the goldens are pinned by test_gpu_parity.py and test_gpu_golden.py."""
    import torch
    from vi_depth_completion_b200 import _torchops
    assert _torchops.ops() is torch.ops.vidc
    w, rgb, depth, normals, g, a = _setup(cuda_device)
    _, y = w.warp_with_gravity_center_aligned(rgb, g, a)
    w.warp_with_gravity_center_aligned(depth, g, a, interp_mode="nearest")
    w.inverse_warp_normal_image_with_gravity_center_aligned(normals, g, a)
    w.unwarp_normals(normals, g, a)
    w.warp_rgbd(rgb, depth, g, a)
    w._build_homography(g, a)
    _, ycl = w.warp_with_gravity_center_aligned(rgb.contiguous(memory_format=torch.channels_last), g, a)
    assert ycl.is_contiguous(memory_format=torch.channels_last) and not ycl.is_contiguous()
    assert y.is_contiguous() and torch.equal(ycl, y)


def test_extension_error_behaviour(cuda_device):
    import torch
    w, rgb, depth, normals, g, a = _setup(cuda_device)
    with pytest.raises(AssertionError):                                # reference :123
        w.warp_with_gravity_center_aligned(rgb[:3], g, a)
    with pytest.raises(AssertionError):                                # reference :224
        w.inverse_warp_normal_image_with_gravity_center_aligned(normals[:2], g, a)
    with pytest.raises(IndexError):                                    # reference :41
        w.warp_with_gravity_center_aligned(rgb, g, a[:1])
    with pytest.raises(RuntimeError):
        w.warp_with_gravity_center_aligned(rgb.double(), g, a)
    with pytest.raises(RuntimeError):
        torch.ops.vidc.warp_forward(rgb.cpu(), g, a, 202., 202., 159.9, 119.9, 0)      # no CPU kernel is registered


def test_torch_compile_fullgraph(cuda_device):
    import torch
    w, rgb, depth, normals, g, a = _setup(cuda_device)

    def path(x, n, gg, aa):
        _, x1 = w.warp_with_gravity_center_aligned(x, gg, aa)
        _, z = w.inverse_warp_normal_image_with_gravity_center_aligned(n * 2.0, gg, aa)
        return x1 + 1.0, torch.nn.functional.normalize(z, dim=1)

    with torch.no_grad():
        want = path(rgb, normals, g, a)
        got = torch.compile(path, fullgraph=True, backend="aot_eager")(rgb, normals, g, a)
    assert torch.equal(want[0], got[0]) and torch.equal(want[1], got[1])


def test_parameters_prepared_once_per_batch(cuda_device):
    """prepare() + warp_rgbd(params=) + unwarp_normals(params=): one per-frame kernel for the batch instead of one per call
    (the reference rebuilds the homographies in every call, :124 and :225).  Same bits as the calls that take I_g / I_a; two
    launches saved per step; the handle is checked (camera, batch, device)."""
    import torch
    from vi_depth_completion_b200 import _cabi
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment
    w, rgb, depth, normals, g, a = _setup(cuda_device, B=5)
    H0, r0, d0, m0 = w.warp_rgbd(rgb, depth, g, a)
    _, z0 = w.unwarp_normals(normals, g, a)
    _, zr0 = w.unwarp_normals(normals, g, a, normalize=False)
    n0 = _cabi.lib().vidc_launch_count()
    p = w.prepare(g, a)
    H1, r1, d1, m1 = w.warp_rgbd(rgb, depth, params=p)
    H2, z1 = w.unwarp_normals(normals, params=p)
    _, zr1 = w.unwarp_normals(normals, params=p, normalize=False)
    assert _cabi.lib().vidc_launch_count() - n0 == 4                    # 1 per-frame kernel + 3 warps
    for x, y in ((H0, H1), (H0, H2), (r0, r1), (d0, d1), (m0, m1), (z0, z1), (zr0, zr1)):
        assert torch.equal(x, y)
    assert depth.dim() == 3 and d1.dim() == 3                            # 3-D depth in, 3-D depth out (:110-112, :153-154)
    d4 = w.warp_rgbd(rgb, depth[:, None], params=p)[2]
    assert d4.dim() == 4 and torch.equal(d4[:, 0], d0)
    with pytest.raises(AssertionError):
        w.warp_rgbd(rgb[:3], depth[:3], params=p)                        # batch of the handle
    with pytest.raises(RuntimeError):
        Warping2DOFAlignment(404., 404., 319.87654, 239.87603).unwarp_normals(normals, params=p)   # another camera
    with pytest.raises(RuntimeError):
        w.unwarp_normals(normals)                                        # neither gravity nor params
    x = rgb.clone().requires_grad_(True)
    out = w.warp_rgbd(x, depth, params=p)
    with pytest.raises(NotImplementedError):
        out[1].sum().backward()
