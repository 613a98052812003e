// kernels_generic.cuh -- generic-stride kernels (any layout / size) and the small caller-side helpers
// Part of libvidc_b200.so (one translation unit, vidc_kernels.cu); compiled with -fmad=false.
#pragma once
#include "device_common.cuh"

namespace vidc_k {

// ------------------------------------------------------------------------------------------
// Forward warp.  MODE_A: interpolation of image A (C_A channels, 1..4); image D (1 channel, optional)
// has its own mode.  ROT: rotate the 3 channels of A by R after sampling (:288, intent of :258-290).
// View: ImgView (fp32) or ImgViewU8 (uint8 frames, every tap through load_tap).
template <int C_A, bool HAS_D, bool ROT, typename View>
__device__ __forceinline__ void
warp_forward_pixel(const vidc_frame_params* __restrict__ prm, CamConst cam,
                   View a, ImgViewOut ya, int mode_a,
                   ImgView d, ImgViewOut yd, int mode_d,
                   unsigned char* __restrict__ mask, unsigned int* __restrict__ coverage) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    const vidc_frame_params* __restrict__ P = prm + b;
    float Hi[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) Hi[k] = __ldg(&P->Hinv[k]);
    const float px_min = __ldg(&P->px_min), py_min = __ldg(&P->py_min);
    const float ikw = __ldg(&P->ikw), ikh = __ldg(&P->ikh);
    const bool live = X < cam.W && Y < cam.H;
    bool m = false;
    if (live) {
        float out_a[C_A];
        {
            float ix, iy;
            forward_coords(Hi, px_min, py_min, ikw, ikh, cam, (float)X, (float)Y, (float)a.w, (float)a.h, ix, iy);
            const typename View::elem* __restrict__ base = a.p + (long long)b * a.sn;
            if (mode_a == VIDC_BILINEAR) {
                const Taps t = bilinear_taps(ix, iy, a.h, a.w, a.sh, a.sw);
#pragma unroll
                for (int c = 0; c < C_A; ++c) out_a[c] = sample_bilinear(base + c * a.sc, t);
            } else if (mode_a == VIDC_BICUBIC) {
                float rx, ry;
                forward_coords_raw(Hi, px_min, py_min, ikw, ikh, cam, (float)X, (float)Y, (float)a.w, (float)a.h, rx, ry);
                const CubicTaps t = bicubic_taps(rx, ry, a.h, a.w);
#pragma unroll
                for (int c = 0; c < C_A; ++c) out_a[c] = sample_bicubic(base + c * a.sc, t, a.sh, a.sw);
            } else {
#pragma unroll
                for (int c = 0; c < C_A; ++c) out_a[c] = sample_nearest(base + c * a.sc, ix, iy, a.h, a.w, a.sh, a.sw);
            }
        }
        if (ROT && C_A == 3) {
            float R[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) R[k] = __ldg(&P->R[k]);
            float z[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) z[c] = fmaf(R[3 * c + 2], out_a[2], fmaf(R[3 * c + 1], out_a[1], fmaf(R[3 * c], out_a[0], 0.0f)));
#pragma unroll
            for (int c = 0; c < 3; ++c) out_a[c] = z[c];
        }
        float* __restrict__ ob = ya.p + (long long)b * ya.sn + Y * ya.sh + X * ya.sw;
#pragma unroll
        for (int c = 0; c < C_A; ++c) ob[c * ya.sc] = out_a[c];
        if (C_A == 3) m = (out_a[0] + out_a[1]) + out_a[2] > 0.01f;       // surface_normal.py:151
        if (HAS_D) {
            float ix, iy;
            forward_coords(Hi, px_min, py_min, ikw, ikh, cam, (float)X, (float)Y, (float)d.w, (float)d.h, ix, iy);
            const float* __restrict__ base = d.p + (long long)b * d.sn;
            float v;
            if (mode_d == VIDC_BILINEAR) {
                const Taps t = bilinear_taps(ix, iy, d.h, d.w, d.sh, d.sw);
                v = sample_bilinear(base, t);
            } else {
                v = sample_nearest(base, ix, iy, d.h, d.w, d.sh, d.sw);
            }
            yd.p[(long long)b * yd.sn + Y * yd.sh + X * yd.sw] = v;
        }
        if (mask) mask[((long long)b * cam.H + Y) * cam.W + X] = m ? 1 : 0;
    }
    if (coverage) {   // warp-shuffle (ballot) reduction, then one shared and one global atomic per CTA
        __shared__ unsigned int cta_count;
        const int tid = threadIdx.y * blockDim.x + threadIdx.x;
        if (tid == 0) cta_count = 0;
        __syncthreads();
        const unsigned int bal = __ballot_sync(0xffffffffu, m);
        if ((tid & 31) == 0 && bal) atomicAdd(&cta_count, __popc(bal));
        __syncthreads();
        if (tid == 0 && cta_count) atomicAdd(coverage + b, cta_count);
    }
}
template <int C_A, bool HAS_D, bool ROT>
__global__ void __launch_bounds__(256)
warp_forward_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam,
                    ImgView a, ImgViewOut ya, int mode_a,
                    ImgView d, ImgViewOut yd, int mode_d,
                    unsigned char* __restrict__ mask, unsigned int* __restrict__ coverage) {
    warp_forward_pixel<C_A, HAS_D, ROT>(prm, cam, a, ya, mode_a, d, yd, mode_d, mask, coverage);
}
// (B,Hin,Win,3) uint8 RGB of vidc_warp_rgbd_u8 where the sheared uint8 kernel does not apply (bilinear RGB, optional depth)
template <bool HAS_D>
__global__ void __launch_bounds__(256)
warp_forward_u8_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam,
                       ImgViewU8 a, ImgViewOut ya, int mode_a,
                       ImgView d, ImgViewOut yd, int mode_d,
                       unsigned char* __restrict__ mask, unsigned int* __restrict__ coverage) {
    warp_forward_pixel<3, HAS_D, false>(prm, cam, a, ya, mode_a, d, yd, mode_d, mask, coverage);
}

// Inverse warp of normals: gather + R^T rotation (+ F.normalize), ref :242-253, surface_normal.py:170
template <bool NORMALIZE>
__global__ void __launch_bounds__(256)
unwarp_normals_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam,
                      ImgView x, ImgViewOut z, unsigned char* __restrict__ valid) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    if (X >= cam.W || Y >= cam.H) return;
    const vidc_frame_params* __restrict__ P = prm + b;
    float Hm[9], R[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) { Hm[k] = __ldg(&P->H[k]); R[k] = __ldg(&P->R[k]); }
    const float px_min = __ldg(&P->px_min), py_min = __ldg(&P->py_min);
    const float kw = __ldg(&P->kw), kh = __ldg(&P->kh);
    float ix, iy;
    inverse_coords(Hm, px_min, py_min, kw, kh, cam, (float)X, (float)Y, (float)x.w, (float)x.h, ix, iy);
    const Taps t = bilinear_taps(ix, iy, x.h, x.w, x.sh, x.sw);
    const float* __restrict__ base = x.p + (long long)b * x.sn;
    const float y0 = sample_bilinear(base, t);
    const float y1 = sample_bilinear(base + x.sc, t);
    const float y2 = sample_bilinear(base + 2 * x.sc, t);
    // z = C_R_Cg.bmm(y), C_R_Cg = R^T: z_c = sum_k R[k][c] y_k, k-ascending FMA chain from a +0
    // accumulator like the GEMM behind bmm (:253) -- the seed decides the sign of a zero result: I * (-0) = +0
    float z0 = fmaf(R[6], y2, fmaf(R[3], y1, fmaf(R[0], y0, 0.0f)));
    float z1 = fmaf(R[7], y2, fmaf(R[4], y1, fmaf(R[1], y0, 0.0f)));
    float z2 = fmaf(R[8], y2, fmaf(R[5], y1, fmaf(R[2], y0, 0.0f)));
    if (NORMALIZE) {   // z / max(||z||, 1e-12); squares summed left to right without FMA
        const float n = clamp_min_eps(sqrtf((z0 * z0 + z1 * z1) + z2 * z2));
        z0 = z0 / n; z1 = z1 / n; z2 = z2 / n;
    }
    float* __restrict__ ob = z.p + (long long)b * z.sn + Y * z.sh + X * z.sw;
    ob[0] = z0; ob[z.sc] = z1; ob[2 * z.sc] = z2;
    if (valid) valid[((long long)b * cam.H + Y) * cam.W + X] = (t.b_nw || t.b_ne || t.b_sw || t.b_se) ? 1 : 0;
}

// image_sampler_forward_inverse (:158-214): both grids, (B,H,W,2) contiguous, aspect guard :178-187
__global__ void __launch_bounds__(256)
sampler_grids_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam,
                     float2* __restrict__ grid, float2* __restrict__ inv_grid) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    if (X >= cam.W || Y >= cam.H) return;
    const vidc_frame_params* __restrict__ P = prm + b;
    const float sigma = __ldg(&P->w_max) / __ldg(&P->h_max);              // :178
    const bool guard = sigma < 0.8f || sigma > 2.2f;                       // :179
    const long long o = ((long long)b * cam.H + Y) * cam.W + X;
    const float Xf = (float)X, Yf = (float)Y;
    float2 g, gi;
    if (guard) {                                                           // :181-186
        g.x = cam.inv_half_w * (Xf - cam.cx);
        g.y = cam.inv_half_h * (Yf - cam.cy);
        gi = g;
    } else {
        const float px_min = __ldg(&P->px_min), py_min = __ldg(&P->py_min);
        {
            const float* Hi = P->Hinv;
            const float px = __ldg(&P->ikw) * Xf + px_min;
            const float py = __ldg(&P->ikh) * Yf + py_min;
            const float u = fmaf(__ldg(Hi + 1), py, __ldg(Hi + 0) * px) + __ldg(Hi + 2);
            const float v = fmaf(__ldg(Hi + 4), py, __ldg(Hi + 3) * px) + __ldg(Hi + 5);
            const float s = fmaf(__ldg(Hi + 7), py, __ldg(Hi + 6) * px) + __ldg(Hi + 8);
            g.x = cam.inv_half_w * (u / s - cam.cx);
            g.y = cam.inv_half_h * (v / s - cam.cy);
        }
        {
            const float* Hm = P->H;
            const float u = fmaf(__ldg(Hm + 1), Yf, __ldg(Hm + 0) * Xf) + __ldg(Hm + 2);
            const float v = fmaf(__ldg(Hm + 4), Yf, __ldg(Hm + 3) * Xf) + __ldg(Hm + 5);
            const float s = fmaf(__ldg(Hm + 7), Yf, __ldg(Hm + 6) * Xf) + __ldg(Hm + 8);
            const float cxp = __ldg(&P->kw) * (u / s - px_min);
            const float cyp = __ldg(&P->kh) * (v / s - py_min);
            gi.x = cam.inv_half_w * (cxp - cam.cx);
            gi.y = cam.inv_half_h * (cyp - cam.cy);
        }
    }
    if (grid) grid[o] = g;
    if (inv_grid) inv_grid[o] = gi;
}

__global__ void guard_rt_kernel(const vidc_frame_params* __restrict__ prm, int B, float* __restrict__ Rt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * 9) return;
    const int b = i / 9, k = i % 9;
    const float sigma = prm[b].w_max / prm[b].h_max;
    const bool guard = sigma < 0.8f || sigma > 2.2f;
    Rt[i] = guard ? ((k % 4 == 0) ? 1.0f : 0.0f) : prm[b].R[3 * (k % 3) + k / 3];
}

// surface_normal.py:151 standalone
__global__ void __launch_bounds__(256)
validity_mask_kernel(ImgView x, unsigned char* __restrict__ mu8, float* __restrict__ mf32,
                     unsigned int* __restrict__ coverage) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    bool m = false;
    if (X < x.w && Y < x.h) {
        const float* __restrict__ p = x.p + (long long)b * x.sn + Y * x.sh + X * x.sw;
        m = (__ldg(p) + __ldg(p + x.sc)) + __ldg(p + 2 * x.sc) > 0.01f;
        const long long o = ((long long)b * x.h + Y) * x.w + X;
        if (mu8) mu8[o] = m ? 1 : 0;
        if (mf32) mf32[o] = m ? 1.0f : 0.0f;
    }
    if (coverage) {
        __shared__ unsigned int cta_count;
        const int tid = threadIdx.y * blockDim.x + threadIdx.x;
        if (tid == 0) cta_count = 0;
        __syncthreads();
        const unsigned int bal = __ballot_sync(0xffffffffu, m);
        if ((tid & 31) == 0 && bal) atomicAdd(&cta_count, __popc(bal));
        __syncthreads();
        if (tid == 0 && cta_count) atomicAdd(coverage + b, cta_count);
    }
}

// F.interpolate(mask, size, 'nearest'): src = min(floor(dst * (float)in / out), in - 1)
__global__ void mask_nearest_kernel(const float* __restrict__ m, int B, int Hin, int Win, int Hout, int Wout,
                                    float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)B * Hout * Wout;
    if (i >= total) return;
    const int x = (int)(i % Wout), y = (int)((i / Wout) % Hout), b = (int)(i / ((long long)Wout * Hout));
    const float sh = (float)Hin / (float)Hout, sw = (float)Win / (float)Wout;
    const int sy = min((int)floorf((float)y * sh), Hin - 1), sx = min((int)floorf((float)x * sw), Win - 1);
    out[i] = __ldg(m + ((long long)b * Hin + sy) * Win + sx);
}

// all pyramid levels of surface_normal.py:153-156 in one launch (row f3); src u8 or f32 mask, f32 outputs
struct PyramidArgs {
    const unsigned char* m8; const float* m32;
    int B, Hin, Win, levels;
    int Ho[4], Wo[4];
    long long begin[5];          // prefix sums of B*Ho*Wo
    float* out[4];
};
__global__ void mask_pyramid_kernel(const __grid_constant__ PyramidArgs a) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.begin[a.levels]) return;
    int l = 0;
#pragma unroll
    for (int k = 1; k < 4; ++k) if (k < a.levels && i >= a.begin[k]) l = k;
    const long long r = i - a.begin[l];
    const int Ho = a.Ho[l], Wo = a.Wo[l];
    const int x = (int)(r % Wo), y = (int)((r / Wo) % Ho), b = (int)(r / ((long long)Wo * Ho));
    const float sh = (float)a.Hin / (float)Ho, sw = (float)a.Win / (float)Wo;
    const int sy = min((int)floorf((float)y * sh), a.Hin - 1), sx = min((int)floorf((float)x * sw), a.Win - 1);
    const long long src = ((long long)b * a.Hin + sy) * a.Win + sx;
    a.out[l][r] = a.m8 ? (a.m8[src] ? 1.0f : 0.0f) : __ldg(a.m32 + src);
}

__global__ void __launch_bounds__(256) normalize3_kernel(ImgView z, ImgViewOut o) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    if (X >= z.w || Y >= z.h) return;
    const float* __restrict__ p = z.p + (long long)b * z.sn + Y * z.sh + X * z.sw;
    const float z0 = __ldg(p), z1 = __ldg(p + z.sc), z2 = __ldg(p + 2 * z.sc);
    const float n = clamp_min_eps(sqrtf((z0 * z0 + z1 * z1) + z2 * z2));
    float* __restrict__ q = o.p + (long long)b * o.sn + Y * o.sh + X * o.sw;
    q[0] = z0 / n; q[o.sc] = z1 / n; q[2 * o.sc] = z2 / n;
}

// Contiguous planes (the common case): four pixels per thread, 128-bit loads and stores, grid-stride over the frame.
// hw4 = H * W / 4; planes are hw4 float4s apart; frames are z_sn / o_sn floats apart.
__global__ void __launch_bounds__(256) normalize3_vec4_kernel(const float* __restrict__ z, long long z_sn, float* __restrict__ o,
                                                              long long o_sn, int hw4) {
    const int b = blockIdx.y;
    const float4* __restrict__ p = reinterpret_cast<const float4*>(z + (long long)b * z_sn);
    float4* __restrict__ q = reinterpret_cast<float4*>(o + (long long)b * o_sn);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw4; i += gridDim.x * blockDim.x) {
        const float4 a0 = __ldg(p + i), a1 = __ldg(p + hw4 + i), a2 = __ldg(p + 2 * hw4 + i);
        float4 r0, r1, r2;
        float n;
        n = clamp_min_eps(sqrtf((a0.x * a0.x + a1.x * a1.x) + a2.x * a2.x)); r0.x = a0.x / n; r1.x = a1.x / n; r2.x = a2.x / n;
        n = clamp_min_eps(sqrtf((a0.y * a0.y + a1.y * a1.y) + a2.y * a2.y)); r0.y = a0.y / n; r1.y = a1.y / n; r2.y = a2.y / n;
        n = clamp_min_eps(sqrtf((a0.z * a0.z + a1.z * a1.z) + a2.z * a2.z)); r0.z = a0.z / n; r1.z = a1.z / n; r2.z = a2.z / n;
        n = clamp_min_eps(sqrtf((a0.w * a0.w + a1.w * a1.w) + a2.w * a2.w)); r0.w = a0.w / n; r1.w = a1.w / n; r2.w = a2.w / n;
        q[i] = r0; q[hw4 + i] = r1; q[2 * hw4 + i] = r2;
    }
}
// surface_normal.py:151 on contiguous planes: four pixels per thread, u8 and / or float mask, coverage by popc
__global__ void __launch_bounds__(256) validity_mask_vec4_kernel(const float* __restrict__ x, long long x_sn, int hw4,
                                                                 unsigned char* __restrict__ mu8, float* __restrict__ mf32,
                                                                 unsigned int* __restrict__ coverage) {
    const int b = blockIdx.y;
    const float4* __restrict__ p = reinterpret_cast<const float4*>(x + (long long)b * x_sn);
    unsigned int cnt = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw4; i += gridDim.x * blockDim.x) {
        const float4 r = __ldg(p + i), g = __ldg(p + hw4 + i), bl = __ldg(p + 2 * hw4 + i);
        const unsigned int m0 = (r.x + g.x) + bl.x > 0.01f, m1 = (r.y + g.y) + bl.y > 0.01f;
        const unsigned int m2 = (r.z + g.z) + bl.z > 0.01f, m3 = (r.w + g.w) + bl.w > 0.01f;
        const long long o4 = (long long)b * hw4 + i;
        if (mu8) reinterpret_cast<unsigned int*>(mu8)[o4] = m0 | (m1 << 8) | (m2 << 16) | (m3 << 24);
        if (mf32) reinterpret_cast<float4*>(mf32)[o4] = make_float4((float)m0, (float)m1, (float)m2, (float)m3);
        cnt += m0 + m1 + m2 + m3;
    }
    if (coverage) {
        __shared__ unsigned int cta_count;
        if (threadIdx.x == 0) cta_count = 0;
        __syncthreads();
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&cta_count, cnt);
        __syncthreads();
        if (threadIdx.x == 0 && cta_count) atomicAdd(coverage + b, cta_count);
    }
}

// normal_utils.py:7-34 in one pass; fp64 block reduction (warp shuffles), one atomic per CTA per stat
__global__ void __launch_bounds__(256)
normal_stats_kernel(ImgView gt, ImgView pred, ImgView mask, int normalize_prediction, double* __restrict__ out) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    double s_ang = 0.0, s_m = 0.0, s_l1 = 0.0, s_cos = 0.0;
    if (X < gt.w && Y < gt.h) {
        const float* __restrict__ pp = pred.p + (long long)b * pred.sn + Y * pred.sh + X * pred.sw;
        const float* __restrict__ pg = gt.p + (long long)b * gt.sn + Y * gt.sh + X * gt.sw;
        const float m = __ldg(mask.p + (long long)b * mask.sn + Y * mask.sh + X * mask.sw);
        const float r0 = __ldg(pp), r1 = __ldg(pp + pred.sc), r2 = __ldg(pp + 2 * pred.sc);
        const float g0 = __ldg(pg), g1 = __ldg(pg + gt.sc), g2 = __ldg(pg + 2 * gt.sc);
        float n0 = r0, n1 = r1, n2 = r2;
        const float nr = sqrtf((r0 * r0 + r1 * r1) + r2 * r2);
        if (normalize_prediction) {
            const float nn = clamp_min_eps(nr);
            n0 = r0 / nn; n1 = r1 / nn; n2 = r2 / nn;
        }
        float dp = (n0 * g0 + n1 * g1) + n2 * g2;
        dp = dp < -1.0f ? -1.0f : dp;                      // torch.clamp keeps NaN (normal_utils.py:12)
        dp = dp > 1.0f ? 1.0f : dp;
        const float ang = (float)((double)acosf(dp) / 3.14159265358979323846 * 180.0);
        s_ang = (double)(ang * m);
        s_m = (double)m;
        s_l1 = fabs((double)(n0 * m) - (double)(g0 * m)) + fabs((double)(n1 * m) - (double)(g1 * m)) +
               fabs((double)(n2 * m) - (double)(g2 * m));
        // F.cosine_similarity(pred, gt, dim=1), eps = 1e-8 on each norm
        const float ng = sqrtf((g0 * g0 + g1 * g1) + g2 * g2);
        s_cos = (double)(((r0 * g0 + r1 * g1) + r2 * g2) / (clamp_min_nan(nr, 1e-8f) * clamp_min_nan(ng, 1e-8f)));
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        s_ang += __shfl_down_sync(0xffffffffu, s_ang, off);
        s_m += __shfl_down_sync(0xffffffffu, s_m, off);
        s_l1 += __shfl_down_sync(0xffffffffu, s_l1, off);
        s_cos += __shfl_down_sync(0xffffffffu, s_cos, off);
    }
    __shared__ double sm[4][8];
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    if ((tid & 31) == 0) { sm[0][tid >> 5] = s_ang; sm[1][tid >> 5] = s_m; sm[2][tid >> 5] = s_l1; sm[3][tid >> 5] = s_cos; }
    __syncthreads();
    if (tid < 4) {
        double t = 0.0;
        const int nw = (blockDim.x * blockDim.y + 31) >> 5;
        for (int w = 0; w < nw; ++w) t += sm[tid][w];
        if (t != 0.0) atomicAdd(out + tid, t);
    }
}

// Backward of the two losses of normal_utils.py w.r.t. pred_normals (the training loss of network_run.py:186,248), one pass.
//   mode 0: compute_normal_vectors_loss_l1, normalize_prediction=True   loss = sum|n^ m - g m| / sum(m)      (:20-34)
//   mode 1: the same with normalize_prediction=False                     (n^ = pred)
//   mode 2: compute_normal_vectors_loss_l2                               loss = -sum(cos_sim(pred, g)) / sum(m) (:7-10, NOT masked)
// stats[1] = sum(mask) from the forward pass (vidc_normal_stats); *grad_loss = upstream gradient of the scalar loss.
// Torch's chain, in torch's order (N = clamped norm, |r| = unclamped norm, q_c = (r_c / N) / N):
//   L1Loss(sum)      -> sign(a - b), with sign(0) = sign(NaN) = 0
//   x / N            -> dx_c = grad_c / N and dN = -sum_c grad_c q_c   (div backward: -grad * ((x / N) / N); N^2 and N^3
//                       are never formed, so nothing overflows before the norm itself does at |r| ~ 1.8e19)
//   F.normalize      -> N = |r|.clamp_min(1e-12): dN reaches the norm only where |r| >= 1e-12 (clamp_min backward)
//   cosine_similarity-> N = |r|.clamp_min_(1e-8) under no_grad: the clamp is invisible to autograd, so dN always reaches
//                       the norm, and the radial term survives for every |r| > 0 (the division uses the clamped norm)
//   vector_norm      -> dr_c += dN * (r_c / |r|), where |r| == 0 gives 0
// The clamps keep NaN (as torch's clamp_min does), so a NaN in pred gives a NaN gradient.  Channels >= 3 of pred get zeros.
__global__ void __launch_bounds__(256)
normal_loss_backward_kernel(ImgView gt, ImgView pred, ImgView mask, int mode, const double* __restrict__ stats,
                            const float* __restrict__ grad_loss, ImgViewOut gp) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    if (X >= gt.w || Y >= gt.h) return;
    const float go = __ldg(grad_loss) / (float)__ldg(stats + 1);
    const float* __restrict__ pp = pred.p + (long long)b * pred.sn + Y * pred.sh + X * pred.sw;
    const float* __restrict__ pg = gt.p + (long long)b * gt.sn + Y * gt.sh + X * gt.sw;
    float* __restrict__ po = gp.p + (long long)b * gp.sn + Y * gp.sh + X * gp.sw;
    const float m = __ldg(mask.p + (long long)b * mask.sn + Y * mask.sh + X * mask.sw);
    const float r[3] = {__ldg(pp), __ldg(pp + pred.sc), __ldg(pp + 2 * pred.sc)};
    const float g[3] = {__ldg(pg), __ldg(pg + gt.sc), __ldg(pg + 2 * gt.sc)};
    const float nr = sqrtf((r[0] * r[0] + r[1] * r[1]) + r[2] * r[2]);
    float dx[3], nc;          // gradient reaching x / N, and the clamped norm N
    float dN = 0.0f;          // gradient reaching the unclamped norm
    if (mode == 2) {
        const float ng = clamp_min_nan(sqrtf((g[0] * g[0] + g[1] * g[1]) + g[2] * g[2]), 1e-8f);
        nc = clamp_min_nan(nr, 1e-8f);
#pragma unroll
        for (int c = 0; c < 3; ++c) dx[c] = -go * (g[c] / ng);
    } else {
        nc = clamp_min_eps(nr);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float n = mode == 0 ? r[c] / nc : r[c];
            const float diff = n * m - g[c] * m;
            const float sg = diff > 0.0f ? 1.0f : (diff < 0.0f ? -1.0f : 0.0f);  // torch.sign: 0 for 0 and for NaN
            dx[c] = go * sg * m;
        }
    }
    if (mode != 1) {
        const float dd = (dx[0] * ((r[0] / nc) / nc) + dx[1] * ((r[1] / nc) / nc)) + dx[2] * ((r[2] / nc) / nc);
        if (mode == 2 || nr >= 1e-12f) dN = -dd;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) po[c * gp.sc] = mode == 1 ? dx[c] : dx[c] / nc + dN * (nr == 0.0f ? 0.0f : r[c] / nr);
    for (int c = 3; c < gp.c; ++c) po[c * gp.sc] = 0.0f;
}

// ---- ToTensor on device (dataset.py:468-471, the data format on the DataLoader side of the path) -----------------------------
// (B,H,W,C) uint8 as PIL decodes it -> (B,C,H,W) float = x / 255.  HBM-bound: C bytes in, 4 C bytes out per pixel.
// RGB fast path: thread -> 4 consecutive pixels = three aligned 32-bit loads, one 128-bit store per plane.
__global__ void __launch_bounds__(256) to_tensor_rgb_u8_kernel(const uint32_t* __restrict__ in, long long hw, float* __restrict__ out) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;            // quad of pixels inside the frame
    if (4 * q >= hw) return;
    const int b = blockIdx.y;
    const uint32_t* __restrict__ src = in + ((long long)b * hw * 3) / 4 + 3 * q;
    const uint32_t w0 = __ldg(src), w1 = __ldg(src + 1), w2 = __ldg(src + 2);        // R0 G0 B0 R1 | G1 B1 R2 G2 | B2 R3 G3 B3
    float* __restrict__ o = out + (long long)b * 3 * hw + 4 * q;
    *reinterpret_cast<float4*>(o) = make_float4(vidc::u8_to_unit(w0 & 255u), vidc::u8_to_unit(w0 >> 24),
                                                vidc::u8_to_unit((w1 >> 16) & 255u), vidc::u8_to_unit((w2 >> 8) & 255u));
    *reinterpret_cast<float4*>(o + hw) = make_float4(vidc::u8_to_unit((w0 >> 8) & 255u), vidc::u8_to_unit(w1 & 255u),
                                                     vidc::u8_to_unit(w1 >> 24), vidc::u8_to_unit((w2 >> 16) & 255u));
    *reinterpret_cast<float4*>(o + 2 * hw) = make_float4(vidc::u8_to_unit((w0 >> 16) & 255u), vidc::u8_to_unit((w1 >> 8) & 255u),
                                                         vidc::u8_to_unit(w2 & 255u), vidc::u8_to_unit(w2 >> 24));
}
// any channel count / size: thread -> one output value
__global__ void __launch_bounds__(256) to_tensor_u8_kernel(const uint8_t* __restrict__ in, long long hw, int C, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;            // pixel inside the frame
    if (i >= hw) return;
    const int b = blockIdx.y;
    const uint8_t* __restrict__ src = in + ((long long)b * hw + i) * C;
    for (int c = 0; c < C; ++c) out[((long long)b * C + c) * hw + i] = vidc::u8_to_unit(src[c]);
}

}  // namespace vidc_k
