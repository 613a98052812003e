// device_common.cuh -- image views, ATen grid_sampler primitives and the exact coordinate chains shared by every kernel
// Part of libvidc_b200.so (one translation unit, vidc_kernels.cu); compiled with -fmad=false.
#pragma once
#include "frame_params.cuh"

namespace vidc_k {

// ------------------------------------------------------------------------------------------
// device-side image view (strides in elements; intra-frame offsets fit 32 bits)
struct ImgView {
    using elem = float;
    const float* __restrict__ p;
    int c, h, w;
    long long sn;
    int sc, sh, sw;
};
// (B,H,W,3) uint8 frames as the loader holds them (vidc_warp_rgbd_u8): element strides (3 H W, 1, 3 W, 3)
struct ImgViewU8 {
    using elem = uint8_t;
    const uint8_t* __restrict__ p;
    int c, h, w;
    long long sn;
    int sc, sh, sw;
};
struct ImgViewOut {
    float* __restrict__ p;
    int c, h, w;
    long long sn;
    int sc, sh, sw;
};

struct CamConst {
    float cx, cy, inv_half_w, inv_half_h;
    int W, H;
};

// norm.clamp_min(1e-12) of F.normalize (torch/nn/functional.py; surface_normal.py:170): unlike fmaxf(), a NaN
// norm stays NaN, so every component of a vector holding one NaN comes out NaN, as in the reference.
__device__ __forceinline__ float clamp_min_eps(float n) { return n < 1e-12f ? 1e-12f : n; }
// torch's clamp_min (x < lo ? lo : x): keeps NaN, unlike fmaxf
__device__ __forceinline__ float clamp_min_nan(float x, float lo) { return x < lo ? lo : x; }

// ATen grid_sampler_2d, align_corners=False: ((g + 1) * size - 1) / 2 with the multiply-subtract
// contracted into one fma, as both the CPU and the CUDA builds of ATen compile it.
__device__ __forceinline__ float unnormalize(float g, float size) {
    return fmaf(g + 1.0f, size, -1.0f) * 0.5f;
}
// GridSampler.cuh:140-147 safe_downgrade_to_int_range
__device__ __forceinline__ float safe_coord(float x) {
    return (x > 2147483646.0f || x < -2147483648.0f || !isfinite(x)) ? -100.0f : x;
}

struct Taps {
    int o_nw, o_ne, o_sw, o_se;      // element offsets inside one channel plane (only valid if in-bounds)
    float w_nw, w_ne, w_sw, w_se;
    bool b_nw, b_ne, b_sw, b_se;
};

__device__ __forceinline__ Taps bilinear_taps(float ix, float iy, int Hin, int Win, int sh, int sw) {
    Taps t;
    const float x0f = floorf(ix), y0f = floorf(iy);
    const float x1f = x0f + 1.0f, y1f = y0f + 1.0f;
    const int x0 = (int)x0f, y0 = (int)y0f, x1 = x0 + 1, y1 = y0 + 1;
    const float wx1 = ix - x0f, wx0 = x1f - ix, wy1 = iy - y0f, wy0 = y1f - iy;
    t.w_nw = wx0 * wy0; t.w_ne = wx1 * wy0; t.w_sw = wx0 * wy1; t.w_se = wx1 * wy1;
    const bool in_x0 = (unsigned)x0 < (unsigned)Win, in_x1 = (unsigned)x1 < (unsigned)Win;
    const bool in_y0 = (unsigned)y0 < (unsigned)Hin, in_y1 = (unsigned)y1 < (unsigned)Hin;
    t.b_nw = in_x0 && in_y0; t.b_ne = in_x1 && in_y0; t.b_sw = in_x0 && in_y1; t.b_se = in_x1 && in_y1;
    t.o_nw = y0 * sh + x0 * sw; t.o_ne = t.o_nw + sw; t.o_sw = t.o_nw + sh; t.o_se = t.o_sw + sw;
    return t;
}

// One tap as fp32: a float element as it is, a uint8 element as ToTensor makes it (x / 255, vidc::u8_to_unit), so a warp
// of uint8 frames gives the bits of the same warp of to_tensor(frames).
__device__ __forceinline__ float load_tap(const float* __restrict__ p) { return __ldg(p); }
__device__ __forceinline__ float load_tap(const uint8_t* __restrict__ p) { return vidc::u8_to_unit(__ldg(p)); }

template <typename T>
__device__ __forceinline__ float sample_bilinear(const T* __restrict__ plane, const Taps& t) {
    const float v_nw = t.b_nw ? load_tap(plane + t.o_nw) : 0.0f;
    const float v_ne = t.b_ne ? load_tap(plane + t.o_ne) : 0.0f;
    const float v_sw = t.b_sw ? load_tap(plane + t.o_sw) : 0.0f;
    const float v_se = t.b_se ? load_tap(plane + t.o_se) : 0.0f;
    // ATen accumulates nw, ne, sw, se with fused multiply-adds; a skipped (out-of-bounds) tap
    // equals adding 0 * w exactly.
    float acc = v_nw * t.w_nw;
    acc = fmaf(v_ne, t.w_ne, acc);
    acc = fmaf(v_sw, t.w_sw, acc);
    acc = fmaf(v_se, t.w_se, acc);
    return acc;
}

template <typename T>
__device__ __forceinline__ float sample_nearest(const T* __restrict__ plane, float ix, float iy,
                                                int Hin, int Win, int sh, int sw) {
    const int xn = (int)rintf(ix), yn = (int)rintf(iy);      // round half to even, as nearbyint
    const bool in = (unsigned)xn < (unsigned)Win && (unsigned)yn < (unsigned)Hin;
    return in ? load_tap(plane + yn * sh + xn * sw) : 0.0f;
}

// ---- bicubic (interp_mode='bicubic', A = -0.75): ATen's cubic convolution as torch 2.11 rounds it on CPU (oracle/warp_oracle.c,
// pinned bit-for-bit against F.grid_sample).  The weights come from the UNCLIPPED coordinate -- a non-finite coordinate gives
// NaN weights and a NaN result in both builds of ATen -- while each tap coordinate goes through safe_downgrade_to_int_range.
__device__ __forceinline__ void bicubic_coefficients(float t, float c[4]) {
    const float A = -0.75f;
    float x = t + 1.0f;
    c[0] = ((A * x - 5.0f * A) * x + 8.0f * A) * x - 4.0f * A;
    x = t;
    c[1] = fmaf(fmaf(A + 2.0f, x, -(A + 3.0f)) * x, x, 1.0f);
    x = 1.0f - t;
    c[2] = fmaf(fmaf(A + 2.0f, x, -(A + 3.0f)) * x, x, 1.0f);
    x = 2.0f - t;
    c[3] = ((A * x - 5.0f * A) * x + 8.0f * A) * x - 4.0f * A;
}
struct CubicTaps {
    float cx[4], cy[4];
    int xi[4], yi[4];          // tap coordinates, already range-checked: -1 = out of bounds
};
__device__ __forceinline__ CubicTaps bicubic_taps(float rx, float ry, int Hin, int Win) {
    CubicTaps t;
    const float x0f = floorf(rx), y0f = floorf(ry);
    bicubic_coefficients(rx - x0f, t.cx);
    bicubic_coefficients(ry - y0f, t.cy);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int xk = (int)safe_coord(x0f + (float)(k - 1)), yk = (int)safe_coord(y0f + (float)(k - 1));
        t.xi[k] = ((unsigned)xk < (unsigned)Win) ? xk : -1;
        t.yi[k] = ((unsigned)yk < (unsigned)Hin) ? yk : -1;
    }
    return t;
}
template <typename T>
__device__ __forceinline__ float sample_bicubic(const T* __restrict__ plane, const CubicTaps& t, int sh, int sw) {
    float rows[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (t.yi[i] >= 0 && t.xi[j] >= 0) ? load_tap(plane + t.yi[i] * sh + t.xi[j] * sw) : 0.0f;
        float acc = fmaf(t.cx[0], v[0], t.cx[1] * v[1]);          // ((c0 v0 + c1 v1) + c2 v2) + c3 v3, first add contracted
        acc = acc + t.cx[2] * v[2];
        acc = acc + t.cx[3] * v[3];
        rows[i] = acc;
    }
    float acc = t.cy[0] * rows[0];                                // FMA chain over the four rows
    acc = fmaf(t.cy[1], rows[1], acc);
    acc = fmaf(t.cy[2], rows[2], acc);
    acc = fmaf(t.cy[3], rows[3], acc);
    return acc;
}

// canvas pixel (X, Y) -> source pixel coordinates of the input image (ref :142-150 + ATen unnormalise)
__device__ __forceinline__ void forward_coords(const float* __restrict__ Hi, float px_min, float py_min,
                                               float ikw, float ikh, const CamConst& cam, float X, float Y,
                                               float Win, float Hin, float& ix, float& iy) {
    const float px = ikw * X + px_min;
    const float py = ikh * Y + py_min;
    // (3,3)@(3,WH) mm: k-ascending FMA chain; fma(h, 1, acc) == acc + h
    const float u = fmaf(Hi[1], py, Hi[0] * px) + Hi[2];
    const float v = fmaf(Hi[4], py, Hi[3] * px) + Hi[5];
    const float s = fmaf(Hi[7], py, Hi[6] * px) + Hi[8];
    const float sx = u / s, sy = v / s;                                    // :146-147
    const float gx = cam.inv_half_w * (sx - cam.cx);                       // :149
    const float gy = cam.inv_half_h * (sy - cam.cy);                       // :150
    ix = safe_coord(unnormalize(gx, Win));
    iy = safe_coord(unnormalize(gy, Hin));
}
// the same without the range clip (bicubic weights use the raw coordinate)
__device__ __forceinline__ void forward_coords_raw(const float* __restrict__ Hi, float px_min, float py_min,
                                                   float ikw, float ikh, const CamConst& cam, float X, float Y,
                                                   float Win, float Hin, float& ix, float& iy) {
    const float px = ikw * X + px_min;
    const float py = ikh * Y + py_min;
    const float u = fmaf(Hi[1], py, Hi[0] * px) + Hi[2];
    const float v = fmaf(Hi[4], py, Hi[3] * px) + Hi[5];
    const float s = fmaf(Hi[7], py, Hi[6] * px) + Hi[8];
    const float sx = u / s, sy = v / s;
    ix = unnormalize(cam.inv_half_w * (sx - cam.cx), Win);
    iy = unnormalize(cam.inv_half_h * (sy - cam.cy), Hin);
}

// camera pixel (X, Y) -> canvas pixel coordinates (ref :242-249 + ATen unnormalise)
__device__ __forceinline__ void inverse_coords(const float* __restrict__ Hm, float px_min, float py_min,
                                               float kw, float kh, const CamConst& cam, float X, float Y,
                                               float Win, float Hin, float& ix, float& iy) {
    const float u = fmaf(Hm[1], Y, Hm[0] * X) + Hm[2];
    const float v = fmaf(Hm[4], Y, Hm[3] * X) + Hm[5];
    const float s = fmaf(Hm[7], Y, Hm[6] * X) + Hm[8];
    const float tx = u / s, ty = v / s;                                    // :245
    const float cxp = kw * (tx - px_min);                                  // :246
    const float cyp = kh * (ty - py_min);                                  // :247
    const float gx = cam.inv_half_w * (cxp - cam.cx);                      // :248
    const float gy = cam.inv_half_h * (cyp - cam.cy);                      // :249
    ix = safe_coord(unnormalize(gx, Win));
    iy = safe_coord(unnormalize(gy, Hin));
}

}  // namespace vidc_k
