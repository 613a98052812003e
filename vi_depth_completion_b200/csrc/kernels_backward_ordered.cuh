// kernels_backward_ordered.cuh -- deterministic gather backward of the two warps (row f4, fixed summation order)
// Part of libvidc_b200.so (one translation unit, vidc_kernels.cu); compiled with -fmad=false.
//
// The scatter kernel of kernels_backward.cuh adds w_tap * g into grad_in with atomicAdd, so the order of the fp32 additions
// changes from run to run.  This kernel computes the same sums in ONE fixed order, the order a serial scatter loop produces:
// every element of grad_in starts at +0 and receives, in output row-major order (Y, then X), the rounded product w_tap * g of
// every output pixel that has it among its in-bounds taps (nearest: the rint tap, contribution g itself), each added with a
// separate rounding.  The coordinates and weights are the forward kernels' bits (forward_coords / inverse_coords /
// bilinear_taps); the inverse warp first rotates g <- R g with the scatter kernel's FMA chain.  tests/harness/backward_scatter.c
// restates it as a plain C loop over the CPU oracle's sampling grids.
//
// Layout: one CTA of 256 threads per 32x32 tile of grad_in and frame; every thread owns the tile column tid & 31 in the rows
// (tid >> 5) + 8 j, j = 0..3, and keeps their (up to 4) channel sums in registers for the whole kernel.  Every element of
// grad_in is written exactly once: no memset, no global atomics.
//   1. Candidate box (thread 0, fp64): the output pixels whose taps can reach the tile are those whose source coordinate lies
//      in the tile's +-1 px window.  The window's corners are mapped back through the exact inverse of the coordinate map (the
//      adjugate of the frame's homography), as the sparse-depth kernel does; their bounding box plus a margin is the candidate
//      box.  A window on which the inverse map has a pole (denominator of mixed sign or ill-conditioned) or that maps to
//      non-finite points takes the whole output plane: correctness never depends on the box being tight, only on it being
//      conservative.
//   2. The box is streamed in row-major chunks of 256 pixels, one per thread: the thread evaluates its pixel's coordinates and
//      weights once, stores them with its (rotated) gradient in shared memory and appends its local index k to the list of
//      its tap origin (x0, y0) (nearest: the rint tap) if that origin lies in the tile's 33x33 origin grid.
//   3. Each owner then merges the lists of its up to four origins -- nw from (x, y), ne from (x-1, y), sw from (x, y-1),
//      se from (x-1, y-1) -- by k, which is the output row-major order within the chunk, and adds in that order.  The result
//      does not depend on the order in which the lists were filled, and the chunks are visited in order, so each element's
//      whole sum runs in output row-major order.  A chunk in which a list overflows its BWO_CAP entries (heavy upsampling) is
//      instead merged by scanning all of its pixels in order: slow but exact.
#pragma once
#include "device_common.cuh"

namespace vidc_k {

constexpr int BWO_TILE = 32, BWO_ORG = BWO_TILE + 1, BWO_NORG = BWO_ORG * BWO_ORG, BWO_CHUNK = 256, BWO_CAP = 8;

struct BwoBox { int x0, y0, w, h; };

__device__ __forceinline__ void adjugate3(const double* m, double* a) {
    a[0] = m[4] * m[8] - m[5] * m[7]; a[1] = m[2] * m[7] - m[1] * m[8]; a[2] = m[1] * m[5] - m[2] * m[4];
    a[3] = m[5] * m[6] - m[3] * m[8]; a[4] = m[0] * m[8] - m[2] * m[6]; a[5] = m[2] * m[3] - m[0] * m[5];
    a[6] = m[3] * m[7] - m[4] * m[6]; a[7] = m[1] * m[6] - m[0] * m[7]; a[8] = m[0] * m[4] - m[1] * m[3];
}

// Output pixels whose source coordinate can fall in the window [qx0 - 1, qx1 + 1] x [qy0 - 1, qy1 + 1] of source pixels.
// Forward warp: source (ix, iy) -> camera pixel -> adj(Hinv) -> canvas point (px, py) -> canvas pixel (px - px_min) / ikw.
// Inverse warp: source = canvas pixel -> point (tx, ty) = cxp / kw + px_min -> adj(H) -> camera pixel.
template <bool INVERSE>
__device__ BwoBox bwo_candidate_box(const vidc_frame_params* __restrict__ P, const CamConst& cam, int Hin, int Win,
                                    int qx0, int qy0, int qx1, int qy1) {
    const BwoBox whole = {0, 0, cam.W, cam.H};
    double M[9], A[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) M[k] = INVERSE ? (double)P->H[k] : (double)P->Hinv[k];
    adjugate3(M, A);
    const double px_min = P->px_min, py_min = P->py_min;
    const double kx = INVERSE ? P->kw : P->ikw, ky = INVERSE ? P->kh : P->ikh;
    double xlo = 1e300, xhi = -1e300, ylo = 1e300, yhi = -1e300, slo = 1e300, shi = -1e300;
    bool ok = true;
    for (int c = 0; c < 4; ++c) {
        const double qx = (c & 1) ? qx1 + 1.0 : qx0 - 1.0, qy = (c & 2) ? qy1 + 1.0 : qy0 - 1.0;
        double a = ((2.0 * qx + 1.0) / Win - 1.0) / cam.inv_half_w + cam.cx;       // un-normalise, then gx -> pixel
        double b = ((2.0 * qy + 1.0) / Hin - 1.0) / cam.inv_half_h + cam.cy;
        if (INVERSE) { a = a / kx + px_min; b = b / ky + py_min; }
        const double t0 = A[6] * a, t1 = A[7] * b;
        const double s = t0 + t1 + A[8];
        double X = (A[0] * a + A[1] * b + A[2]) / s, Y = (A[3] * a + A[4] * b + A[5]) / s;
        if (!INVERSE) { X = (X - px_min) / kx; Y = (Y - py_min) / ky; }
        ok = ok && fabs(s) > 1e-3 * (fabs(t0) + fabs(t1) + fabs(A[8])) && fabs(X) < 1e9 && fabs(Y) < 1e9;   // also rejects NaN
        xlo = fmin(xlo, X); xhi = fmax(xhi, X); ylo = fmin(ylo, Y); yhi = fmax(yhi, Y);
        slo = fmin(slo, s); shi = fmax(shi, s);
    }
    if (!(ok && (slo > 0.0 || shi < 0.0))) return whole;                    // pole inside the window: every output pixel
    const double mx = 2.0 + 1e-3 * fmax(fabs(xlo), fabs(xhi)), my = 2.0 + 1e-3 * fmax(fabs(ylo), fabs(yhi));
    int X0 = (int)floor(xlo - mx), X1 = (int)ceil(xhi + mx), Y0 = (int)floor(ylo - my), Y1 = (int)ceil(yhi + my);
    X0 = X0 < 0 ? 0 : X0; Y0 = Y0 < 0 ? 0 : Y0;
    X1 = X1 > cam.W - 1 ? cam.W - 1 : X1; Y1 = Y1 > cam.H - 1 ? cam.H - 1 : Y1;
    if (X1 < X0 || Y1 < Y0) { const BwoBox empty = {0, 0, 0, 0}; return empty; }
    const BwoBox b = {X0, Y0, X1 - X0 + 1, Y1 - Y0 + 1};
    return b;
}

template <bool INVERSE>
__global__ void __launch_bounds__(256, 3)            // 3 CTAs (24 warps) per SM: <= 85 registers
warp_backward_ordered_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam, ImgView gy /* (B,C,H,W) grad of the output */,
                             int C, int mode, float* __restrict__ gx, long long gx_sn, int gx_sc, int Hin, int Win) {
    __shared__ int cnt[2][BWO_NORG];                   // list lengths per tap origin, double-buffered by chunk parity
    __shared__ unsigned char lst[BWO_NORG][BWO_CAP];   // chunk-local pixel indices k per tap origin (insertion order arbitrary)
    __shared__ short org[BWO_CHUNK];                   // tap-origin slot of chunk pixel k, -1 = outside the tile's origin grid
    __shared__ float wk[4][BWO_CHUNK];                 // w_nw, w_ne, w_sw, w_se of chunk pixel k
    __shared__ float gk[4][BWO_CHUNK];                 // its (rotated) upstream gradient, per channel
    __shared__ int ovf[2];                             // a list of this chunk overflowed
    __shared__ BwoBox box;
    const int tid = threadIdx.x, b = blockIdx.z;
    const int qx0 = blockIdx.x * BWO_TILE, qy0 = blockIdx.y * BWO_TILE;
    const vidc_frame_params* __restrict__ P = prm + b;
    for (int i = tid; i < 2 * BWO_NORG; i += 256) (&cnt[0][0])[i] = 0;
    if (tid < 2) ovf[tid] = 0;
    if (tid == 0)
        box = bwo_candidate_box<INVERSE>(P, cam, Hin, Win, qx0, qy0, min(qx0 + BWO_TILE - 1, Win - 1), min(qy0 + BWO_TILE - 1, Hin - 1));
    float M[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) M[k] = INVERSE ? __ldg(&P->H[k]) : __ldg(&P->Hinv[k]);
    const float px_min = __ldg(&P->px_min), py_min = __ldg(&P->py_min);
    const float kx = INVERSE ? __ldg(&P->kw) : __ldg(&P->ikw), ky = INVERSE ? __ldg(&P->kh) : __ldg(&P->ikh);
    float R[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) R[k] = INVERSE ? __ldg(&P->R[k]) : 0.0f;
    const bool bil = mode == VIDC_BILINEAR;
    const float* __restrict__ gframe = gy.p + (long long)b * gy.sn;
    __syncthreads();
    const int bx0 = box.x0, by0 = box.y0, bw = box.w, n = box.w * box.h;

    const int lx = tid & 31;
    float acc[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[j][c] = 0.0f;
    int prev_o = -1;
    for (int c0 = 0, it = 0; c0 < n; c0 += BWO_CHUNK, ++it) {
        const int par = it & 1;
        // 2. this thread's pixel of the chunk
        const int i = c0 + tid;
        int o = -1;
        if (i < n) {
            const int r = i / bw;
            const int X = bx0 + (i - r * bw), Y = by0 + r;
            float ix, iy;
            if (INVERSE) inverse_coords(M, px_min, py_min, kx, ky, cam, (float)X, (float)Y, (float)Win, (float)Hin, ix, iy);
            else forward_coords(M, px_min, py_min, kx, ky, cam, (float)X, (float)Y, (float)Win, (float)Hin, ix, iy);
            const int ox = bil ? (int)floorf(ix) : (int)rintf(ix), oy = bil ? (int)floorf(iy) : (int)rintf(iy);
            if (ox >= qx0 - 1 && ox <= qx0 + BWO_TILE - 1 && oy >= qy0 - 1 && oy <= qy0 + BWO_TILE - 1) {
                o = (oy - qy0 + 1) * BWO_ORG + (ox - qx0 + 1);
                if (bil) {
                    const Taps t = bilinear_taps(ix, iy, Hin, Win, Win, 1);
                    wk[0][tid] = t.w_nw; wk[1][tid] = t.w_ne; wk[2][tid] = t.w_sw; wk[3][tid] = t.w_se;
                }
                const float* __restrict__ g = gframe + Y * gy.sh + X * gy.sw;
                float gv[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) gv[c] = c < C ? __ldg(g + c * gy.sc) : 0.0f;
                if (INVERSE) {   // z = R^T y  =>  dL/dy = R dL/dz (kernels_backward.cuh)
                    const float a0 = gv[0], a1 = gv[1], a2 = gv[2];
                    gv[0] = fmaf(R[2], a2, fmaf(R[1], a1, fmaf(R[0], a0, 0.0f)));
                    gv[1] = fmaf(R[5], a2, fmaf(R[4], a1, fmaf(R[3], a0, 0.0f)));
                    gv[2] = fmaf(R[8], a2, fmaf(R[7], a1, fmaf(R[6], a0, 0.0f)));
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) gk[c][tid] = gv[c];
            }
        }
        org[tid] = (short)o;
        if (prev_o >= 0) cnt[par ^ 1][prev_o] = 0;       // the previous chunk's lists are consumed: empty them for chunk it + 1
        if (tid == 0) ovf[par ^ 1] = 0;
        if (o >= 0) {
            const int s = atomicAdd(&cnt[par][o], 1);
            if (s < BWO_CAP) lst[o][s] = (unsigned char)tid;
            else ovf[par] = 1;
        }
        prev_o = o;
        __syncthreads();
        // 3. owners: merge by k and add in that order
        const bool over = ovf[par] != 0;
        const int nk = min(BWO_CHUNK, n - c0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ly = (tid >> 5) + 8 * j;
            if (qx0 + lx >= Win || qy0 + ly >= Hin) continue;
            const int o_nw = (ly + 1) * BWO_ORG + lx + 1;
            const int os[4] = {o_nw, o_nw - 1, o_nw - BWO_ORG, o_nw - BWO_ORG - 1};   // origins of the nw, ne, sw, se taps
            const int ntap = bil ? 4 : 1;
            if (!over) {
                int m[4], tot = 0;
#pragma unroll
                for (int t = 0; t < 4; ++t) { m[t] = t < ntap ? cnt[par][os[t]] : 0; tot += m[t]; }
                // the k of the four lists are distinct (a pixel has one tap origin): take them smallest first
                int cur = -1;
                for (int rnk = 0; rnk < tot; ++rnk) {
                    int best = BWO_CHUNK, bt = 0;
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        for (int s = 0; s < m[t]; ++s) {
                            const int k = lst[os[t]][s];
                            if (k > cur && k < best) { best = k; bt = t; }
                        }
                    const float w = bil ? wk[bt][best] : 1.0f;
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (c < C) acc[j][c] = __fadd_rn(acc[j][c], bil ? __fmul_rn(w, gk[c][best]) : gk[c][best]);
                    cur = best;
                }
            } else {
                for (int k = 0; k < nk; ++k) {
                    const int ok = org[k];
                    int bt = -1;
#pragma unroll
                    for (int t = 0; t < 4; ++t) if (t < ntap && ok == os[t]) bt = t;
                    if (bt < 0) continue;
                    const float w = bil ? wk[bt][k] : 1.0f;
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (c < C) acc[j][c] = __fadd_rn(acc[j][c], bil ? __fmul_rn(w, gk[c][k]) : gk[c][k]);
                }
            }
        }
        __syncthreads();
    }
    float* __restrict__ out = gx + (long long)b * gx_sn;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int x = qx0 + lx, y = qy0 + (tid >> 5) + 8 * j;
        if (x >= Win || y >= Hin) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c)
            if (c < C) out[(long long)c * gx_sc + y * Win + x] = acc[j][c];
    }
}

}  // namespace vidc_k
