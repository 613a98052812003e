// kernels_grad_params.cuh -- gradient of the two warps with respect to the per-frame parameters, and its chain to I_g / I_a
// Part of libvidc_b200.so (one translation unit, vidc_kernels.cu); compiled with -fmad=false.
//
// In the reference the sampling grid of F.grid_sample is built from H^-1 (forward warp, :142-150) or H (inverse warp,
// :242-249) and the canvas scale with differentiable ops, so autograd sends a gradient into the frame parameters and on to
// I_g and I_a.  Per output pixel this kernel takes ATen's grid_sampler_2d_backward grid gradient (bilinear, zeros padding,
// align_corners=False)
//     gix = sum_c g_c [(ne - nw)(y1 - iy) + (se - sw)(iy - y0)]      giy = sum_c g_c [(sw - nw)(x1 - ix) + (se - ne)(ix - x0)]
// (an out-of-bounds tap reads 0) and applies the chain ix -> gx -> (sx = u / s) -> (u, v, s) -> the parameters:
//   forward (any C):  dL/dHinv (9), dL/dpx_min, dL/dpy_min, dL/dikw, dL/dikh       (P = (ikw X + px_min, ikh Y + py_min, 1))
//   inverse (C = 3):  dL/dH (9), dL/dpx_min, dL/dpy_min, dL/dkw, dL/dkh, dL/dR (9) (z = R^T n: dL/dn = R g, dL/dR[k][c] += n_k g_c)
// The coordinates are the forward kernels' bits (forward_coords / inverse_coords); a non-finite coordinate contributes 0.
// 'nearest' has a zero grid gradient, as in ATen: the host writes zeros and launches nothing.
//
// Order (bit-reproducible, independent of the frame's batch position and of the stream; no global atomics):
//   1. one CTA of 256 threads per 32x32 output tile and frame; thread (lx, ly) takes rows ly, ly + 8, ly + 16, ly + 24 of
//      column lx in that order and adds each pixel's terms to fp64 sums;
//   2. a fixed shuffle tree per warp, then warps 0..7 in order: the tile's partial sums go to the tile's own slot of the
//      caller's scratch (vidc_warp_backward_params_scratch_bytes);
//   3. grad_params_reduce_kernel adds each frame's tiles in row-major tile order, in fp64, and rounds once to fp32.
#pragma once
#include "device_common.cuh"
#include "frame_params_grad.cuh"

namespace vidc_k {

constexpr int GP_TILE = 32, GP_NV = 22;     // slots: [0..8] Hinv | H, [9] px_min, [10] py_min, [11] ikw | kw, [12] ikh | kh, [13..21] R

template <bool INVERSE>
__global__ void __launch_bounds__(256)
warp_grad_params_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam, ImgView x /* forward's input */,
                        ImgView gy /* grad of the forward's output */, int C, double* __restrict__ partial) {
    constexpr int NV = INVERSE ? GP_NV : 13;
    __shared__ double red[8][NV];
    const int tid = threadIdx.x, lx = tid & 31, wid = tid >> 5, b = blockIdx.z;
    const vidc_frame_params* __restrict__ P = prm + b;
    float M[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) M[k] = INVERSE ? __ldg(&P->H[k]) : __ldg(&P->Hinv[k]);
    const float px_min = __ldg(&P->px_min), py_min = __ldg(&P->py_min);
    const float kx = INVERSE ? __ldg(&P->kw) : __ldg(&P->ikw), ky = INVERSE ? __ldg(&P->kh) : __ldg(&P->ikh);
    float R[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = INVERSE ? __ldg(&P->R[k]) : 0.0f;
    const float Winf = (float)x.w, Hinf = (float)x.h;
    const float* __restrict__ xf = x.p + (long long)b * x.sn;
    const float* __restrict__ gf = gy.p + (long long)b * gy.sn;
    double acc[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) acc[k] = 0.0;

    const int X = blockIdx.x * GP_TILE + lx;
    for (int j = 0; j < 4; ++j) {
        const int Y = blockIdx.y * GP_TILE + wid + 8 * j;
        if (X >= cam.W || Y >= cam.H) continue;
        float ix, iy;
        if (INVERSE) inverse_coords(M, px_min, py_min, kx, ky, cam, (float)X, (float)Y, Winf, Hinf, ix, iy);
        else forward_coords(M, px_min, py_min, kx, ky, cam, (float)X, (float)Y, Winf, Hinf, ix, iy);
        // the intermediate values of the same chain (identical expressions: the compiler shares them)
        const float qx = INVERSE ? (float)X : kx * (float)X + px_min, qy = INVERSE ? (float)Y : ky * (float)Y + py_min;
        const float u = fmaf(M[1], qy, M[0] * qx) + M[2];
        const float v = fmaf(M[4], qy, M[3] * qx) + M[5];
        const float s = fmaf(M[7], qy, M[6] * qx) + M[8];
        const float tx = u / s, ty = v / s;
        if (!(fabsf(tx) < INFINITY && fabsf(ty) < INFINITY && ix != -100.0f && iy != -100.0f)) continue;   // non-finite: 0
        const Taps t = bilinear_taps(ix, iy, x.h, x.w, x.sh, x.sw);
        const float x0f = floorf(ix), y0f = floorf(iy);
        const float wx1 = ix - x0f, wx0 = (x0f + 1.0f) - ix, wy1 = iy - y0f, wy0 = (y0f + 1.0f) - iy;
        const float* __restrict__ gp = gf + Y * gy.sh + X * gy.sw;
        float gix = 0.0f, giy = 0.0f;
        if (INVERSE) {
            float n[3], gz[3], ax[3], ay[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float* __restrict__ pl = xf + c * x.sc;
                const float nw = t.b_nw ? __ldg(pl + t.o_nw) : 0.0f, ne = t.b_ne ? __ldg(pl + t.o_ne) : 0.0f;
                const float sw = t.b_sw ? __ldg(pl + t.o_sw) : 0.0f, se = t.b_se ? __ldg(pl + t.o_se) : 0.0f;
                gz[c] = __ldg(gp + c * gy.sc);
                n[c] = fmaf(se, t.w_se, fmaf(sw, t.w_sw, fmaf(ne, t.w_ne, nw * t.w_nw)));      // the forward's sample
                ax[c] = (ne - nw) * wy0 + (se - sw) * wy1;
                ay[c] = (sw - nw) * wx0 + (se - ne) * wx1;
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {                                   // dL/dn = R g
                const float dn = fmaf(R[3 * k + 2], gz[2], fmaf(R[3 * k + 1], gz[1], R[3 * k] * gz[0]));
                gix = fmaf(dn, ax[k], gix);
                giy = fmaf(dn, ay[k], giy);
            }
#pragma unroll
            for (int k = 0; k < 3; ++k)
#pragma unroll
                for (int c = 0; c < 3; ++c) acc[13 + 3 * k + c] += (double)n[k] * (double)gz[c];
        } else {
            for (int c = 0; c < C; ++c) {
                const float* __restrict__ pl = xf + c * x.sc;
                const float nw = t.b_nw ? __ldg(pl + t.o_nw) : 0.0f, ne = t.b_ne ? __ldg(pl + t.o_ne) : 0.0f;
                const float sw = t.b_sw ? __ldg(pl + t.o_sw) : 0.0f, se = t.b_se ? __ldg(pl + t.o_se) : 0.0f;
                const float g = __ldg(gp + c * gy.sc);
                gix = fmaf(g, (ne - nw) * wy0 + (se - sw) * wy1, gix);
                giy = fmaf(g, (sw - nw) * wx0 + (se - ne) * wx1, giy);
            }
        }
        if (gix == 0.0f && giy == 0.0f) continue;
        // ix = ((gx + 1) W - 1) / 2,  gx = ihw (t - cx)  [inverse: t = k (tx - min)]
        double dtx = (double)gix * (0.5 * Winf) * cam.inv_half_w, dty = (double)giy * (0.5 * Hinf) * cam.inv_half_h;
        if (INVERSE) {
            acc[11] += dtx * ((double)tx - px_min); acc[12] += dty * ((double)ty - py_min);
            dtx *= kx; dty *= ky;
            acc[9] -= dtx; acc[10] -= dty;
        }
        const double is = 1.0 / (double)s;
        const double du = dtx * is, dv = dty * is, ds = -(dtx * tx + dty * ty) * is;
        acc[0] += du * qx; acc[1] += du * qy; acc[2] += du;
        acc[3] += dv * qx; acc[4] += dv * qy; acc[5] += dv;
        acc[6] += ds * qx; acc[7] += ds * qy; acc[8] += ds;
        if (!INVERSE) {   // (qx, qy) = (ikw X + px_min, ikh Y + py_min)
            const double dqx = du * M[0] + dv * M[3] + ds * M[6], dqy = du * M[1] + dv * M[4] + ds * M[7];
            acc[9] += dqx; acc[10] += dqy; acc[11] += dqx * X; acc[12] += dqy * Y;
        }
    }
    // fixed reduction tree: lanes, then warps in order
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        double v = acc[k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lx == 0) red[wid][k] = v;
    }
    __syncthreads();
    if (tid < NV) {
        double v = red[0][tid];
#pragma unroll
        for (int w = 1; w < 8; ++w) v += red[w][tid];
        const int tile = blockIdx.y * gridDim.x + blockIdx.x, ntiles = gridDim.x * gridDim.y;
        partial[((long long)b * ntiles + tile) * GP_NV + tid] = v;
    }
}

// one CTA per frame, thread k: slot k of every tile of the frame in tile order -> the field's gradient
__global__ void grad_params_reduce_kernel(const double* __restrict__ partial, int ntiles, int inverse,
                                          vidc_frame_params* __restrict__ out) {
    const int b = blockIdx.x, k = threadIdx.x;
    float* o = reinterpret_cast<float*>(out + b);
    if (k >= 48) return;
    const int NV = inverse ? GP_NV : 13;
    // field offsets in vidc_frame_params (floats): H 0, R 9, Hinv 18, px_min 27, py_min 28, kw 29, kh 30, ikw 31, ikh 32
    int slot = -1;
    if (inverse) {
        if (k < 9) slot = k; else if (k < 18) slot = 13 + (k - 9); else if (k >= 27 && k <= 30) slot = 9 + (k - 27);
    } else {
        if (k >= 18 && k < 27) slot = k - 18; else if (k == 27 || k == 28) slot = 9 + (k - 27); else if (k == 31 || k == 32) slot = 11 + (k - 31);
    }
    double v = 0.0;
    if (slot >= 0 && slot < NV)
        for (int t = 0; t < ntiles; ++t) v += partial[((long long)b * ntiles + t) * GP_NV + slot];
    o[k] = (float)v;
}

// one thread per frame: the adjoint of frame_params_from_gravity (frame_params_grad.cuh)
__global__ void frame_params_backward_kernel(vidc_camera cam, const float* __restrict__ Ig, const float* __restrict__ Ia, int B,
                                             const vidc_frame_params* __restrict__ gparams, const float* __restrict__ gH,
                                             float* __restrict__ gIg, float* __restrict__ gIa) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    const float g[3] = {Ig[3 * i], Ig[3 * i + 1], Ig[3 * i + 2]};
    const float a[3] = {Ia[3 * i], Ia[3 * i + 1], Ia[3 * i + 2]};
    vidc::frame_params_from_gravity_backward(cam, g, a, gparams[i], gH ? gH + 9 * i : nullptr, gIg + 3 * i, gIa + 3 * i);
}

}  // namespace vidc_k
