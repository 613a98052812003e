"""The C-ABI library loads on a CPU-only box and exports every symbol include/vidc_b200.h declares.
No device work is issued here."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "vidc_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(vidc_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound():
    from vi_depth_completion_b200 import _cabi
    lib = _cabi.lib()
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/vidc_b200.h but not exported"
    assert set(names) == set(_cabi.EXPORTED_SYMBOLS), "ctypes binding and header disagree"
    assert lib.vidc_abi_version() == 3


def test_struct_layouts_match_header():
    from vi_depth_completion_b200 import _cabi
    assert ctypes.sizeof(_cabi.VidcCamera) == 4 * (2 + 9 + 9 + 4 + 2)
    assert ctypes.sizeof(_cabi.VidcImage) == 8 + 16 + 32
    assert _cabi.FRAME_PARAMS_FLOATS * 4 == 192


def test_camera_init_and_argument_errors():
    from vi_depth_completion_b200 import _cabi
    lib = _cabi.lib()
    cam = _cabi.VidcCamera()
    assert lib.vidc_camera_init(202.0, 202.0, 159.93827, 119.938015, ctypes.byref(cam)) == _cabi.VIDC_OK
    assert (cam.W, cam.H) == (320, 240)
    assert lib.vidc_camera_init(0.0, 202.0, 159.9, 119.9, ctypes.byref(cam)) == _cabi.VIDC_ERR_INVALID_ARGUMENT
    assert b"intrinsics" in lib.vidc_last_error()
    with pytest.raises(RuntimeError):
        _cabi.check(_cabi.VIDC_ERR_INVALID_ARGUMENT)
    with pytest.raises(AssertionError):
        _cabi.check(_cabi.VIDC_ERR_BATCH_MISMATCH)


def test_drop_in_class_has_the_reference_signatures():
    import inspect
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment as Wd
    sig = lambda f: str(inspect.signature(f))
    assert sig(Wd.__init__) == "(self, fx=288.935305, fy=288.935305, cx=159.93827, cy=119.938015)"
    assert sig(Wd._build_homography) == "(self, I_g, I_a)"
    assert sig(Wd.warp_with_gravity_center_aligned) == "(self, x, I_g, I_a, interp_mode='bilinear')"
    assert sig(Wd.image_sampler_forward_inverse) == "(self, I_g, I_a)"
    assert sig(Wd.inverse_warp_normal_image_with_gravity_center_aligned) == "(self, x, I_g, I_a)"
    assert sig(Wd.warp_normal_image_with_gravity_center_aligned) == "(self, x, I_g, I_a, interp_mode='bilinear')"
    assert sig(Wd.warp_with_homography) == "(self, x, Cg_H_C)"
    w = Wd()
    assert (int(w.W), int(w.H)) == (320, 240)


def test_no_cpu_fallback():
    import torch
    from vi_depth_completion_b200.warping_2dof_alignment import Warping2DOFAlignment as Wd
    w = Wd()
    g = torch.tensor([[0.0, 1.0, 0.0]])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        w.warp_with_gravity_center_aligned(torch.zeros(1, 3, 240, 320), g, g)
    with pytest.raises(RuntimeError):
        w._build_homography(g, g)


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: no product source may import, include or load anything from it."""
    pkg = os.path.join(ROOT, "vi_depth_completion_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"(from|import)\s+oracle|#include\s+\".*oracle|libwarp_oracle", text), f


def test_torch_extension_builds_and_registers_its_operators():
    """The thin torch C++ extension in front of the C ABI (csrc/torch_ops.cpp): loads on a CPU-only box, registers the
    operators with CUDA and Meta kernels; shapes come out of the Meta kernels without a GPU, with the canvas of vidc_camera_init
    and the workspace of vidc_workspace_bytes (at least one frame, as the CUDA kernels allocate it)."""
    import torch
    from vi_depth_completion_b200 import _cabi, build as vb
    torch.ops.load_library(vb.build_torch_ops())
    lib = _cabi.lib()
    # 320x240, 640x480 and 300x201 (a width that is not a multiple of the 32-pixel tile, an odd height)
    for intr in ((202., 202., 159.93827, 119.938015), (404., 404., 319.87654, 239.87603), (190., 190., 150., 100.5)):
        cam = _cabi.VidcCamera()
        assert lib.vidc_camera_init(*intr, ctypes.byref(cam)) == _cabi.VIDC_OK
        Hc, Wc = cam.H, cam.W
        for B in (0, 1, 5):
            x = torch.empty(B, 3, 200, 300, device="meta")
            g = torch.empty(B, 3, device="meta")
            H, y = torch.ops.vidc.warp_forward(x, g, g, *intr, 0)
            assert H.shape == (B, 3, 3) and y.shape == (B, 3, Hc, Wc)
            H, z = torch.ops.vidc.unwarp_normals(x, g, g, *intr, True)
            assert H.shape == (B, 3, 3) and z.shape == (B, 3, Hc, Wc)
            outs = torch.ops.vidc.warp_rgbd(x, x[:, :1], g, g, *intr, 1)
            assert [tuple(o.shape) for o in outs] == [(B, 3, 3), (B, 3, Hc, Wc), (B, 1, Hc, Wc), (B, 1, Hc, Wc)]
            assert outs[3].dtype == torch.uint8
            assert [tuple(m.shape) for m in torch.ops.vidc.build_homography(g, g, *intr)] == [(B, 3, 3)] * 3
            # parameters prepared once per batch: the Meta workspace has the size the library asks for
            ws, H = torch.ops.vidc.frame_params(g, g, *intr)
            assert ws.numel() * 4 == lib.vidc_workspace_bytes(ctypes.byref(cam), max(B, 1)) and H.shape == (B, 3, 3)
            outs = torch.ops.vidc.warp_rgbd_prepared(x, x[:, :1], ws, *intr, 0)
            assert [tuple(o.shape) for o in outs] == [(B, 3, Hc, Wc), (B, 1, Hc, Wc), (B, 1, Hc, Wc)]
            assert torch.ops.vidc.unwarp_normals_prepared(x, ws, *intr, True).shape == (B, 3, Hc, Wc)
    # intrinsics vidc_camera_init rejects are rejected by the Meta kernels too, as by the CUDA kernels
    x, g = torch.empty(2, 3, 240, 320, device="meta"), torch.empty(2, 3, device="meta")
    bad = (202., 202., 0., 119.938015)
    calls = (lambda: torch.ops.vidc.warp_forward(x, g, g, *bad, 0), lambda: torch.ops.vidc.unwarp_normals(x, g, g, *bad, True),
             lambda: torch.ops.vidc.warp_rgbd(x, x[:, :1], g, g, *bad, 0), lambda: torch.ops.vidc.build_homography(g, g, *bad),
             lambda: torch.ops.vidc.frame_params(g, g, *bad))
    for call in calls:
        with pytest.raises(RuntimeError, match="intrinsics"):
            call()


def test_torch_extension_is_required(monkeypatch, tmp_path):
    """The hot entry points have no second route: a missing or unloadable _vidc_torch_ops.so raises and names the fix."""
    from vi_depth_completion_b200 import _torchops
    monkeypatch.setattr(_torchops, "_ops", None)
    monkeypatch.setattr(_torchops, "LIB_PATH", str(tmp_path / "_vidc_torch_ops.so"))
    with pytest.raises(RuntimeError, match=r"python -m vi_depth_completion_b200\.build`"):
        _torchops.ops()
    (tmp_path / "_vidc_torch_ops.so").write_bytes(b"")
    with pytest.raises(RuntimeError, match="--force"):
        _torchops.ops()
