"""Meta kernel of the uint8 forward warp operator (vidc::warp_rgbd_u8): the shapes and dtypes torch.compile traces with, on a
box without a GPU, for every argument set."""
import torch


def test_warp_rgbd_u8_meta_shapes_and_dtypes_for_every_argument_set():
    from vi_depth_completion_b200 import build as vb
    torch.ops.load_library(vb.build_torch_ops())
    intr = (202., 202., 159.93827, 119.938015)                     # 320x240 canvas
    rgb = torch.empty(2, 200, 300, 3, dtype=torch.uint8, device="meta")
    depth = torch.empty(2, 1, 200, 300, device="meta")
    g = torch.empty(2, 3, device="meta")
    H, rgb_w, depth_w, mask, cov = torch.ops.vidc.warp_rgbd_u8(rgb, depth, g, g, None, *intr, 0, True, False)
    assert [tuple(o.shape) for o in (H, rgb_w, depth_w, mask)] == [(2, 3, 3), (2, 3, 240, 320), (2, 1, 240, 320), (2, 1, 240, 320)]
    assert [o.dtype for o in (H, rgb_w, depth_w, mask)] == [torch.float32, torch.float32, torch.float32, torch.uint8]
    assert rgb_w.is_contiguous() and cov is None
    ws, _ = torch.ops.vidc.frame_params(g, g, *intr)
    H, rgb_w, depth_w, mask, cov = torch.ops.vidc.warp_rgbd_u8(rgb, depth, None, None, ws, *intr, 1, True, False)
    assert H is None and cov is None
    assert [tuple(o.shape) for o in (rgb_w, depth_w, mask)] == [(2, 3, 240, 320), (2, 1, 240, 320), (2, 1, 240, 320)]
    assert [o.dtype for o in (rgb_w, depth_w, mask)] == [torch.float32, torch.float32, torch.uint8]
    # no depth, no mask, coverage counts: in both forms
    for src, Hs in (((g, g, None), (2, 3, 3)), ((None, None, ws), None)):
        H, rgb_w, depth_w, mask, cov = torch.ops.vidc.warp_rgbd_u8(rgb, None, *src, *intr, 0, False, True)
        assert (None if H is None else tuple(H.shape)) == Hs and depth_w is None and mask is None
        assert rgb_w.shape == (2, 3, 240, 320) and rgb_w.dtype == torch.float32 and rgb_w.is_contiguous()
        assert cov.shape == (2,) and cov.dtype == torch.int32
