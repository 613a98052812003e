"""Meta kernels of the uint8 forward warp operators (vidc::warp_rgbd_u8, vidc::warp_rgbd_u8_prepared): the shapes and dtypes
torch.compile traces with, on a box without a GPU."""
import torch


def test_warp_rgbd_u8_meta_shapes_and_dtypes():
    from vi_depth_completion_b200 import build as vb
    torch.ops.load_library(vb.build_torch_ops())
    intr = (202., 202., 159.93827, 119.938015)                     # 320x240 canvas
    rgb = torch.empty(2, 200, 300, 3, dtype=torch.uint8, device="meta")
    depth = torch.empty(2, 1, 200, 300, device="meta")
    g = torch.empty(2, 3, device="meta")
    H, rgb_w, depth_w, mask = torch.ops.vidc.warp_rgbd_u8(rgb, depth, g, g, *intr, 0)
    assert [tuple(o.shape) for o in (H, rgb_w, depth_w, mask)] == [(2, 3, 3), (2, 3, 240, 320), (2, 1, 240, 320), (2, 1, 240, 320)]
    assert [o.dtype for o in (H, rgb_w, depth_w, mask)] == [torch.float32, torch.float32, torch.float32, torch.uint8]
    assert rgb_w.is_contiguous()
    ws, _ = torch.ops.vidc.frame_params(g, g, *intr)
    rgb_w, depth_w, mask = torch.ops.vidc.warp_rgbd_u8_prepared(rgb, depth, ws, *intr, 1)
    assert [tuple(o.shape) for o in (rgb_w, depth_w, mask)] == [(2, 3, 240, 320), (2, 1, 240, 320), (2, 1, 240, 320)]
    assert [o.dtype for o in (rgb_w, depth_w, mask)] == [torch.float32, torch.float32, torch.uint8]
