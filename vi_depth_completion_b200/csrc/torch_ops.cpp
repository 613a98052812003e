// torch_ops.cpp -- the thin torch C++ extension in front of the C ABI (include/vidc_b200.h).
//
// BASELINE.json north star: "calling into hand-written CUDA kernels through a thin torch C++ extension".  This file is that
// extension: TORCH_LIBRARY operators (namespace `vidc`) for the hot entry points of Warping2DOFAlignment
// (networks/warping_2dof_alignment.py:108-156, :216-255, :35-58 of the reference) -- argument checks with TORCH_CHECK (a
// torch RuntimeError, as the reference's own failures are), outputs allocated with ATen, kernels enqueued on
// at::cuda::getCurrentCUDAStream() under a CUDAGuard of the input's device -- plus Meta kernels, so the operators trace under
// torch.compile(fullgraph=True).  No arithmetic lives here: every operator is one call into libvidc_b200.so.  The fused operators
// take every argument set of their C entry point: the per-frame parameters from I_g / I_a or from a workspace frame_params
// filled, and None for an input or output the caller leaves out.
// Built in-tree by vi_depth_completion_b200/build.py into _vidc_torch_ops.so and loaded with torch.ops.load_library.
#include <ATen/ATen.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>

#include <optional>
#include <tuple>

#include "../../include/vidc_b200.h"

namespace {

vidc_camera make_camera(double fx, double fy, double cx, double cy) {
    vidc_camera cam;
    const int rc = vidc_camera_init(fx, fy, cx, cy, &cam);
    TORCH_CHECK(rc == VIDC_OK, "vidc_b200: ", vidc_last_error());
    return cam;
}

void check_status(int rc) {
    if (rc == VIDC_OK) return;
    // the reference's `assert x.shape[0] == I_g.shape[0]` (:123, :224) -- the Python wrapper turns the prefix into AssertionError
    TORCH_CHECK(rc != VIDC_ERR_BATCH_MISMATCH, "vidc_b200 batch mismatch: ", vidc_last_error());
    TORCH_CHECK(false, "vidc_b200: ", vidc_last_error(), " (status ", rc, ")");
}

void check_f32_cuda(const at::Tensor& t, const char* name) {
    TORCH_CHECK(t.is_cuda(), name, ": expected a CUDA tensor (this module has no CPU fallback), got device ", t.device());
    TORCH_CHECK(t.scalar_type() == at::kFloat, name, ": expected scalar type Float but found ", t.scalar_type());
}

vidc_image image_of(const at::Tensor& t) {
    vidc_image im;
    im.data = t.data_ptr<float>();
    im.n = (int32_t)t.size(0); im.c = (int32_t)t.size(1); im.h = (int32_t)t.size(2); im.w = (int32_t)t.size(3);
    im.sn = t.stride(0); im.sc = t.stride(1); im.sh = t.stride(2); im.sw = t.stride(3);
    return im;
}

// I_g / I_a as the kernels read them: (B, 3) contiguous fp32 on x's device, equal batch sizes (:38-43 of the reference)
std::tuple<at::Tensor, at::Tensor> gravity(const at::Tensor& I_g, const at::Tensor& I_a, const at::Device& dev) {
    check_f32_cuda(I_g, "I_g");
    check_f32_cuda(I_a, "I_a");
    TORCH_CHECK(I_g.device() == dev && I_a.device() == dev, "I_g / I_a must live on ", dev, ", got ", I_g.device(), " / ", I_a.device());
    const int64_t B = I_g.size(0), Ba = I_a.size(0);
    TORCH_CHECK(I_g.numel() == 3 * B && I_a.numel() == 3 * Ba, "I_g / I_a: expected 3 components per frame");
    TORCH_CHECK_INDEX(Ba >= B, "index ", Ba, " is out of bounds for dimension 0 with size ", Ba, " (I_a has ", Ba, " frames, I_g has ", B, ")");
    TORCH_CHECK(Ba == B, "I_a has ", Ba, " frames but I_g has ", B, ": batch dimensions of I_a @ I_g must match (ref :43)");
    return {I_g.reshape({B, 3}).contiguous(), I_a.reshape({Ba, 3}).contiguous()};
}

at::Tensor workspace(const vidc_camera& cam, int64_t B, const at::TensorOptions& opt) {
    const size_t bytes = std::max<size_t>(vidc_workspace_bytes(&cam, (int32_t)std::max<int64_t>(B, 1)), sizeof(vidc_frame_params));
    return at::empty({(int64_t)((bytes + 3) / 4)}, opt.dtype(at::kFloat));
}

// outputs adopt the input's memory format (NCHW or channels-last), on the canvas size
at::Tensor canvas_like(const at::Tensor& x, const vidc_camera& cam) {
    const bool cl = x.size(1) > 1 && x.is_contiguous(at::MemoryFormat::ChannelsLast) && !x.is_contiguous();
    return at::empty({x.size(0), x.size(1), cam.H, cam.W}, x.options(), cl ? at::MemoryFormat::ChannelsLast : at::MemoryFormat::Contiguous);
}
// the uint8 validity mask of the fused forward warps and validity plane of the inverse warp: one plane per frame of x
at::Tensor mask_canvas(const at::Tensor& x, const vidc_camera& cam) {
    return at::empty({x.size(0), 1, cam.H, cam.W}, x.options().dtype(at::kByte));
}

using OptTensor = std::optional<at::Tensor>;
template <class T = float>
T* data_or_null(const OptTensor& t) { return t ? t->data_ptr<T>() : nullptr; }

void check_params(const at::Tensor& ws, const vidc_camera& cam, int64_t B, const at::Device& dev) {
    check_f32_cuda(ws, "params");
    TORCH_CHECK(ws.device() == dev, "params must live on ", dev, ", got ", ws.device());
    TORCH_CHECK(ws.is_contiguous() && (size_t)ws.numel() * 4 >= vidc_workspace_bytes(&cam, (int32_t)std::max<int64_t>(B, 1)),
                "params: not a workspace prepared by prepare() for ", B, " frames of this camera");
}

// The fused operators take their per-frame parameters from I_g and I_a or from a workspace frame_params filled: exactly one
// of the two.  Cg_H_C is an output of the first form only (CUDA and Meta kernels alike).
OptTensor homographies(const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params, const at::TensorOptions& opt) {
    TORCH_CHECK(I_g.has_value() == I_a.has_value() && I_g.has_value() != params.has_value(),
                "pass either I_g and I_a or params (a workspace filled by frame_params)");
    return I_g ? OptTensor(at::empty({I_g->size(0), 3, 3}, opt)) : std::nullopt;
}

// The same choice as the C call takes it, once homographies() has checked it: the (B,3) gravity the kernels read and a fresh
// workspace, or d_Ig = d_Ia = NULL and the prepared workspace, whose batch must be x's.
struct Frames {
    OptTensor g, a;
    at::Tensor ws;
    int32_t B;
    vidc_frame_params* prm() const { return reinterpret_cast<vidc_frame_params*>(ws.data_ptr<float>()); }
};
Frames frames(const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params, const vidc_camera& cam, const at::Tensor& x) {
    if (params) {
        check_params(*params, cam, x.size(0), x.device());
        return {std::nullopt, std::nullopt, *params, (int32_t)x.size(0)};
    }
    auto [g, a] = gravity(*I_g, *I_a, x.device());
    return {g, a, workspace(cam, g.size(0), g.options()), (int32_t)g.size(0)};
}

// ---- warp_with_gravity_center_aligned (:108-156), 4-D input ------------------------------------------------------------------
std::tuple<at::Tensor, at::Tensor> warp_forward(const at::Tensor& x, const at::Tensor& I_g, const at::Tensor& I_a, double fx, double fy,
                                                double cx, double cy, int64_t mode) {
    check_f32_cuda(x, "x");
    TORCH_CHECK(x.dim() == 4, "x: expected a 4-D tensor, got ", x.dim(), "-D");
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    const c10::cuda::CUDAGuard guard(x.device());
    auto [g, a] = gravity(I_g, I_a, x.device());
    at::Tensor y = canvas_like(x, cam);
    at::Tensor Hm = at::empty({g.size(0), 3, 3}, x.options());
    at::Tensor ws = workspace(cam, g.size(0), x.options());
    const vidc_image xi = image_of(x), yi = image_of(y);
    check_status(vidc_warp_forward(&cam, &xi, g.data_ptr<float>(), a.data_ptr<float>(), (int32_t)g.size(0), (vidc_interp)mode,
                                   reinterpret_cast<vidc_frame_params*>(ws.data_ptr<float>()), Hm.data_ptr<float>(), &yi,
                                   at::cuda::getCurrentCUDAStream().stream()));
    return {Hm, y};
}

// ---- inverse_warp_normal_image_with_gravity_center_aligned (:216-255) [+ F.normalize of surface_normal.py:170] -----------
// (Cg_H_C, z, valid): the (B,1,H,W) uint8 validity plane only when asked for
using UnwarpOut = std::tuple<OptTensor, at::Tensor, OptTensor>;
UnwarpOut unwarp_outputs(const at::Tensor& x, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params, const vidc_camera& cam,
                         bool with_valid) {
    TORCH_CHECK(x.dim() == 4, "x: expected a 4-D tensor, got ", x.dim(), "-D");
    return {homographies(I_g, I_a, params, x.options()), canvas_like(x, cam), with_valid ? OptTensor(mask_canvas(x, cam)) : std::nullopt};
}
UnwarpOut unwarp_normals(const at::Tensor& x, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params, double fx, double fy,
                         double cx, double cy, bool normalize, bool with_valid) {
    check_f32_cuda(x, "x");
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    const c10::cuda::CUDAGuard guard(x.device());
    UnwarpOut out = unwarp_outputs(x, I_g, I_a, params, cam, with_valid);
    const auto& [H, z, valid] = out;
    const Frames f = frames(I_g, I_a, params, cam, x);
    const vidc_image xi = image_of(x), zi = image_of(z);
    check_status(vidc_unwarp_normals(&cam, &xi, data_or_null(f.g), data_or_null(f.a), f.B, normalize ? 1 : 0, f.prm(), data_or_null(H), &zi,
                                     data_or_null<uint8_t>(valid), at::cuda::getCurrentCUDAStream().stream()));
    return out;
}

// ---- fused forward warp of RGB + depth + validity mask (additive entry point): float RGB (vidc_warp_rgbd) or (B,h,w,3)
// uint8 frames as the loader decodes them (vidc_warp_rgbd_u8), whose RGB comes out as NCHW float32 ------------------------------
// (Cg_H_C, rgb_w, depth_w, mask, coverage): depth_w, the (B,1,H,W) uint8 mask and the (B,) int32 coverage only when asked for
using RgbdOut = std::tuple<OptTensor, at::Tensor, OptTensor, OptTensor, OptTensor>;
RgbdOut rgbd_outputs(const at::Tensor& rgb, const at::Tensor& rgb_w, const OptTensor& depth, const OptTensor& I_g, const OptTensor& I_a,
                     const OptTensor& params, const vidc_camera& cam, bool with_mask, bool with_coverage) {
    return {homographies(I_g, I_a, params, rgb_w.options()), rgb_w, depth ? OptTensor(canvas_like(*depth, cam)) : std::nullopt,
            with_mask ? OptTensor(mask_canvas(rgb, cam)) : std::nullopt,
            with_coverage ? OptTensor(at::empty({rgb.size(0)}, rgb.options().dtype(at::kInt))) : std::nullopt};
}
// the CUDA kernel of both once the RGB is checked: `entry` is the C entry point with its RGB arguments bound
template <class Entry>
RgbdOut fused_rgbd(const vidc_camera& cam, const at::Tensor& rgb, const at::Tensor& rgb_w, const OptTensor& depth, const OptTensor& I_g,
                   const OptTensor& I_a, const OptTensor& params, int64_t depth_mode, bool with_mask, bool with_coverage, Entry entry) {
    if (depth) {
        check_f32_cuda(*depth, "x_depth");
        TORCH_CHECK(depth->dim() == 4, "x_depth: expected (B,1,h,w), got ", depth->dim(), "-D");
        TORCH_CHECK(depth->device() == rgb.device(), "x_depth must live on ", rgb.device(), ", got ", depth->device());
    }
    const c10::cuda::CUDAGuard guard(rgb.device());
    RgbdOut out = rgbd_outputs(rgb, rgb_w, depth, I_g, I_a, params, cam, with_mask, with_coverage);
    const auto& [H, rgb_out, depth_w, mask, cov] = out;
    const Frames f = frames(I_g, I_a, params, cam, rgb);
    vidc_image di{}, dwi{};
    if (depth) {
        di = image_of(*depth);
        dwi = image_of(*depth_w);
    }
    const vidc_image rwi = image_of(rgb_out);
    check_status(entry(depth ? &di : nullptr, data_or_null(f.g), data_or_null(f.a), f.B, (vidc_interp)depth_mode, f.prm(), data_or_null(H),
                       &rwi, depth ? &dwi : nullptr, data_or_null<uint8_t>(mask), reinterpret_cast<uint32_t*>(data_or_null<int32_t>(cov)),
                       at::cuda::getCurrentCUDAStream().stream()));
    return out;
}
RgbdOut warp_rgbd(const at::Tensor& rgb, const OptTensor& depth, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params,
                  double fx, double fy, double cx, double cy, int64_t depth_mode, bool with_mask, bool with_coverage) {
    check_f32_cuda(rgb, "x_rgb");
    TORCH_CHECK(rgb.dim() == 4, "warp_rgbd: expected (B,3,h,w) RGB, got ", rgb.dim(), "-D");
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    const vidc_image ri = image_of(rgb);
    return fused_rgbd(cam, rgb, canvas_like(rgb, cam), depth, I_g, I_a, params, depth_mode, with_mask, with_coverage,
                      [&](auto... rest) { return vidc_warp_rgbd(&cam, &ri, rest...); });
}
void check_u8_frames(const at::Tensor& rgb) {
    TORCH_CHECK(rgb.is_cuda(), "x_rgb: expected a CUDA tensor (this module has no CPU fallback), got device ", rgb.device());
    TORCH_CHECK(rgb.scalar_type() == at::kByte, "x_rgb: expected scalar type Byte but found ", rgb.scalar_type());
    TORCH_CHECK(rgb.dim() == 4 && rgb.size(3) == 3, "x_rgb: expected (B,h,w,3) uint8 frames, got ", rgb.sizes());
    TORCH_CHECK(rgb.is_contiguous(), "x_rgb: expected contiguous (B,h,w,3) frames");
}
at::Tensor rgb_canvas_u8(const at::Tensor& rgb, const vidc_camera& cam) {
    return at::empty({rgb.size(0), 3, cam.H, cam.W}, rgb.options().dtype(at::kFloat));
}
RgbdOut warp_rgbd_u8(const at::Tensor& rgb, const OptTensor& depth, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params,
                     double fx, double fy, double cx, double cy, int64_t depth_mode, bool with_mask, bool with_coverage) {
    check_u8_frames(rgb);
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    return fused_rgbd(cam, rgb, rgb_canvas_u8(rgb, cam), depth, I_g, I_a, params, depth_mode, with_mask, with_coverage, [&](auto... rest) {
        return vidc_warp_rgbd_u8(&cam, rgb.data_ptr<uint8_t>(), (int32_t)rgb.size(0), (int32_t)rgb.size(1), (int32_t)rgb.size(2), rest...);
    });
}

// ---- parameters prepared once per batch and shared by both directions (vidc_frame_params_prepare) ---------------------------------
std::tuple<at::Tensor, at::Tensor> frame_params(const at::Tensor& I_g, const at::Tensor& I_a, double fx, double fy, double cx, double cy) {
    check_f32_cuda(I_g, "I_g");
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    const c10::cuda::CUDAGuard guard(I_g.device());
    auto [g, a] = gravity(I_g, I_a, I_g.device());
    at::Tensor ws = workspace(cam, g.size(0), g.options());
    at::Tensor Hm = at::empty({g.size(0), 3, 3}, g.options());
    check_status(vidc_frame_params_prepare(&cam, g.data_ptr<float>(), a.data_ptr<float>(), (int32_t)g.size(0),
                                           reinterpret_cast<vidc_frame_params*>(ws.data_ptr<float>()), Hm.data_ptr<float>(),
                                           at::cuda::getCurrentCUDAStream().stream()));
    return {ws, Hm};
}

// ---- _build_homography (:35-58) ------------------------------------------------------------------------------------------------
std::tuple<at::Tensor, at::Tensor, at::Tensor> build_homography(const at::Tensor& I_g, const at::Tensor& I_a, double fx, double fy,
                                                                double cx, double cy) {
    check_f32_cuda(I_g, "I_g");
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    const c10::cuda::CUDAGuard guard(I_g.device());
    auto [g, a] = gravity(I_g, I_a, I_g.device());
    at::Tensor out = at::empty({3, g.size(0), 3, 3}, g.options());
    float* p = out.data_ptr<float>();
    const int64_t n = g.size(0) * 9;
    check_status(vidc_build_homography(&cam, g.data_ptr<float>(), a.data_ptr<float>(), (int32_t)g.size(0), p, p + n, p + 2 * n,
                                       at::cuda::getCurrentCUDAStream().stream()));
    return {out[0], out[1], out[2]};
}

// ---- Meta kernels: shapes only (torch.compile / FakeTensor).  The canvas comes from vidc_camera_init and the workspace from
// vidc_workspace_bytes, as in the CUDA kernels, so both allocate the same sizes and reject the same intrinsics ---------------------
std::tuple<at::Tensor, at::Tensor> warp_forward_meta(const at::Tensor& x, const at::Tensor& I_g, const at::Tensor&, double fx, double fy,
                                                     double cx, double cy, int64_t) {
    TORCH_CHECK(x.dim() == 4, "x: expected a 4-D tensor, got ", x.dim(), "-D");
    return {at::empty({I_g.size(0), 3, 3}, x.options()), canvas_like(x, make_camera(fx, fy, cx, cy))};
}
UnwarpOut unwarp_normals_meta(const at::Tensor& x, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params, double fx, double fy,
                              double cx, double cy, bool, bool with_valid) {
    return unwarp_outputs(x, I_g, I_a, params, make_camera(fx, fy, cx, cy), with_valid);
}
RgbdOut warp_rgbd_meta(const at::Tensor& rgb, const OptTensor& depth, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params,
                       double fx, double fy, double cx, double cy, int64_t, bool with_mask, bool with_coverage) {
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    return rgbd_outputs(rgb, canvas_like(rgb, cam), depth, I_g, I_a, params, cam, with_mask, with_coverage);
}
RgbdOut warp_rgbd_u8_meta(const at::Tensor& rgb, const OptTensor& depth, const OptTensor& I_g, const OptTensor& I_a, const OptTensor& params,
                          double fx, double fy, double cx, double cy, int64_t, bool with_mask, bool with_coverage) {
    const vidc_camera cam = make_camera(fx, fy, cx, cy);
    return rgbd_outputs(rgb, rgb_canvas_u8(rgb, cam), depth, I_g, I_a, params, cam, with_mask, with_coverage);
}
std::tuple<at::Tensor, at::Tensor> frame_params_meta(const at::Tensor& I_g, const at::Tensor&, double fx, double fy, double cx, double cy) {
    return {workspace(make_camera(fx, fy, cx, cy), I_g.size(0), I_g.options()), at::empty({I_g.size(0), 3, 3}, I_g.options())};
}
std::tuple<at::Tensor, at::Tensor, at::Tensor> build_homography_meta(const at::Tensor& I_g, const at::Tensor&, double fx, double fy, double cx,
                                                                     double cy) {
    make_camera(fx, fy, cx, cy);
    auto t = [&] { return at::empty({I_g.size(0), 3, 3}, I_g.options()); };
    return {t(), t(), t()};
}

}  // namespace

TORCH_LIBRARY(vidc, m) {
    m.def("warp_forward(Tensor x, Tensor I_g, Tensor I_a, float fx, float fy, float cx, float cy, int mode) -> (Tensor, Tensor)");
    m.def("unwarp_normals(Tensor x, Tensor? I_g, Tensor? I_a, Tensor? params, float fx, float fy, float cx, float cy, bool normalize, "
          "bool with_valid) -> (Tensor?, Tensor, Tensor?)");
    m.def("warp_rgbd(Tensor rgb, Tensor? depth, Tensor? I_g, Tensor? I_a, Tensor? params, float fx, float fy, float cx, float cy, "
          "int depth_mode, bool with_mask, bool with_coverage) -> (Tensor?, Tensor, Tensor?, Tensor?, Tensor?)");
    m.def("warp_rgbd_u8(Tensor rgb, Tensor? depth, Tensor? I_g, Tensor? I_a, Tensor? params, float fx, float fy, float cx, float cy, "
          "int depth_mode, bool with_mask, bool with_coverage) -> (Tensor?, Tensor, Tensor?, Tensor?, Tensor?)");
    m.def("build_homography(Tensor I_g, Tensor I_a, float fx, float fy, float cx, float cy) -> (Tensor, Tensor, Tensor)");
    m.def("frame_params(Tensor I_g, Tensor I_a, float fx, float fy, float cx, float cy) -> (Tensor, Tensor)");
}
TORCH_LIBRARY_IMPL(vidc, CUDA, m) {
    m.impl("warp_forward", &warp_forward);
    m.impl("unwarp_normals", &unwarp_normals);
    m.impl("warp_rgbd", &warp_rgbd);
    m.impl("warp_rgbd_u8", &warp_rgbd_u8);
    m.impl("build_homography", &build_homography);
    m.impl("frame_params", &frame_params);
}
TORCH_LIBRARY_IMPL(vidc, Meta, m) {
    m.impl("warp_forward", &warp_forward_meta);
    m.impl("unwarp_normals", &unwarp_normals_meta);
    m.impl("warp_rgbd", &warp_rgbd_meta);
    m.impl("warp_rgbd_u8", &warp_rgbd_u8_meta);
    m.impl("build_homography", &build_homography_meta);
    m.impl("frame_params", &frame_params_meta);
}
