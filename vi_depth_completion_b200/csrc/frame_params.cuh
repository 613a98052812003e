// frame_params.cuh -- per-frame rotation / homography / canvas-scale parameters.
//
// Restates, with the exact fp32 roundings of the reference executed on CPU (see exact_math.cuh and
// DESIGN.md "accumulate schemes"), networks/warping_2dof_alignment.py:
//   :35-58    _build_homography           (q = g x a, q4 = cos(atan2(|q|, a.g)/2), R, H, Hinv)
//   :125-140  corner projection, bbox, 4:3-fit scale  (repeated at :168-194 and :226-240)
// One thread computes one frame; ~150 fp32 ops, one fp64 cosine.  No host synchronisation
// (the reference performs dozens of device->host reads per frame in this block).
#pragma once
#include "exact_math.cuh"
#include "../../include/vidc_b200.h"

namespace vidc {

// torch.max / torch.min over a 1-D tensor propagate NaN
VIDC_HD float tmax(float a, float b) { return (a != a) ? a : ((b != b) ? b : (a > b ? a : b)); }
VIDC_HD float tmin(float a, float b) { return (a != a) ? a : ((b != b) ? b : (a < b ? a : b)); }

// ref :125-140 given H.  corners: (0,0), (W-1,0), (0,H-1), (W-1,H-1), homogeneous (ref :18)
VIDC_HD void frame_scale(const vidc_camera& cam, const float* Hm, vidc_frame_params& p) {
    const float Wm = (float)(cam.W - 1), Hmm = (float)(cam.H - 1);
    const float cxs[4] = {0.0f, Wm, 0.0f, Wm};
    const float cys[4] = {0.0f, 0.0f, Hmm, Hmm};
    float px[4], py[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const float c0 = dot3_021(Hm[0], Hm[1], Hm[2], cxs[j], cys[j], 1.0f);
        const float c1 = dot3_021(Hm[3], Hm[4], Hm[5], cxs[j], cys[j], 1.0f);
        const float c2 = dot3_021(Hm[6], Hm[7], Hm[8], cxs[j], cys[j], 1.0f);
        px[j] = c0 / c2;                                                    // :126
        py[j] = c1 / c2;
    }
    const float px_max = tmax(tmax(tmax(px[0], px[1]), px[2]), px[3]);      // :127-130
    const float px_min = tmin(tmin(tmin(px[0], px[1]), px[2]), px[3]);
    const float py_max = tmax(tmax(tmax(py[0], py[1]), py[2]), py[3]);
    const float py_min = tmin(tmin(tmin(py[0], py[1]), py[2]), py[3]);
    const float h_max = py_max - py_min;                                    // :132
    const float w_max = px_max - px_min;                                    // :133
    const float Wf = (float)cam.W, Hf = (float)cam.H;
    float kw, kh;
    // python `scalar / tensor` is tensor.reciprocal() * scalar: two roundings
    if (w_max > (4.0f * h_max) / 3.0f) {                                    // :135
        kw = (1.0f / w_max) * Wf;                                           // :136
        kh = (1.0f / ((3.0f * w_max) / 4.0f)) * Hf;                         // :137
    } else {
        kh = (1.0f / h_max) * Hf;                                           // :139
        kw = (1.0f / ((4.0f * h_max) / 3.0f)) * Wf;                         // :140
    }
    p.px_min = px_min; p.py_min = py_min;
    p.kw = kw; p.kh = kh;
    p.ikw = (1.0f / kw) * 1.0f;                                             // "1./kw" :142
    p.ikh = (1.0f / kh) * 1.0f;                                             // "1./kh" :143
    p.w_max = w_max; p.h_max = h_max;
}

// ref :35-58 followed by :125-140
VIDC_HD void frame_params_from_gravity(const vidc_camera& cam, const float* g, const float* a,
                                       vidc_frame_params& p) {
    // :41-42  q = (-[a]x) g  (bmm, mul+add)
    float q0 = dot3_muladd(-0.0f, a[2], -a[1], g[0], g[1], g[2]);
    float q1 = dot3_muladd(-a[2], -0.0f, a[0], g[0], g[1], g[2]);
    float q2 = dot3_muladd(a[1], -a[0], -0.0f, g[0], g[1], g[2]);
    const float d = dot3_muladd(a[0], a[1], a[2], g[0], g[1], g[2]);        // :43
    float ss = q0 * q0;                                                     // :44 norm(dim=1)
    ss = fmaf(q1, q1, ss);
    ss = fmaf(q2, q2, ss);
    const float n = sqrtf(ss);
    const float q4 = mkl_cosf_ha(0.5f * glibc_atan2f(n, d));                // :48
    const float two_q4 = 2.0f * q4;
    q0 = q0 / two_q4; q1 = q1 / two_q4; q2 = q2 / two_q4;                   // :51
    const float S[9] = {0.0f, -q2, q1, q2, 0.0f, -q0, -q1, q0, 0.0f};       // :52
    float* R = p.R;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float I3 = (r == c) ? 1.0f : 0.0f;
            const float t1 = two_q4 * S[3 * r + c];
            const float t2 = dot3_fma(2.0f * S[3 * r], 2.0f * S[3 * r + 1], 2.0f * S[3 * r + 2],
                                      S[c], S[3 + c], S[6 + c]);            // (2.*S) @ S
            R[3 * r + c] = (I3 + t1) + t2;                                  // :53-54
        }
    float KR[9], KRt[9];
    const float* K = cam.K;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            KR[3 * r + c]  = dot3_muladd(K[3 * r], K[3 * r + 1], K[3 * r + 2], R[c], R[3 + c], R[6 + c]);
            KRt[3 * r + c] = dot3_muladd(K[3 * r], K[3 * r + 1], K[3 * r + 2], R[3 * c], R[3 * c + 1], R[3 * c + 2]);
        }
    const float* Ki = cam.Kinv;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            p.H[3 * r + c]    = dot3_fma(KR[3 * r], KR[3 * r + 1], KR[3 * r + 2], Ki[c], Ki[3 + c], Ki[6 + c]);   // :55
            p.Hinv[3 * r + c] = dot3_fma(KRt[3 * r], KRt[3 * r + 1], KRt[3 * r + 2], Ki[c], Ki[3 + c], Ki[6 + c]); // :56-57
        }
    frame_scale(cam, p.H, p);
}

// Conservative 'this 32x32 canvas tile lies entirely outside the source footprint' (kernels_params.cuh explains why it is
// safe; forward warp with input and canvas of the same size).  Not part of any result: it only decides which CTAs may
// write zeros without computing coordinates.
VIDC_HD bool tile_certainly_exterior(const vidc_frame_params& p, const vidc_camera& cam, int tx, int ty) {
    const float Wf = (float)cam.W, Hf = (float)cam.H;
    const float X[2] = {(float)(tx * 32), fminf((float)(tx * 32 + 31), Wf - 1.0f)};
    const float Y[2] = {(float)(ty * 32), fminf((float)(ty * 32 + 31), Hf - 1.0f)};
    float ix_lo = 3.0e38f, ix_hi = -3.0e38f, iy_lo = 3.0e38f, iy_hi = -3.0e38f, s_lo = 3.0e38f, s_hi = -3.0e38f;
    bool ok = true;
    for (int c = 0; c < 4; ++c) {
        const float px = p.ikw * X[c & 1] + p.px_min, py = p.ikh * Y[c >> 1] + p.py_min;
        const float t0 = p.Hinv[6] * px, t1 = p.Hinv[7] * py;
        const float s = t0 + t1 + p.Hinv[8];
        const float u = p.Hinv[0] * px + p.Hinv[1] * py + p.Hinv[2];
        const float v = p.Hinv[3] * px + p.Hinv[4] * py + p.Hinv[5];
        ok = ok && fabsf(s) > 1e-3f * (fabsf(t0) + fabsf(t1) + fabsf(p.Hinv[8]));
        const float ix = ((u / s - cam.cx) * cam.inv_half_w + 1.0f) * Wf * 0.5f - 0.5f;
        const float iy = ((v / s - cam.cy) * cam.inv_half_h + 1.0f) * Hf * 0.5f - 0.5f;
        ok = ok && fabsf(ix) < 1e30f && fabsf(iy) < 1e30f;          // also rejects NaN
        ix_lo = fminf(ix_lo, ix); ix_hi = fmaxf(ix_hi, ix); iy_lo = fminf(iy_lo, iy); iy_hi = fmaxf(iy_hi, iy);
        s_lo = fminf(s_lo, s); s_hi = fmaxf(s_hi, s);
    }
    ok = ok && (s_lo > 0.0f || s_hi < 0.0f);
    const float mx = 4.0f + 2e-3f * fmaxf(fabsf(ix_lo), fabsf(ix_hi)), my = 4.0f + 2e-3f * fmaxf(fabsf(iy_lo), fabsf(iy_hi));
    return ok && (ix_hi < -1.0f - mx || ix_lo > Wf + mx || iy_hi < -1.0f - my || iy_lo > Hf + my);
}

// Source-image bounding box of forward canvas tile (tx, ty) -- the rows an L2 prefetch one wave ahead should ask for
// (kernels_shear.cuh).  A hint only, from the same four mapped corners as the exterior test: out = {x0, y0, w, h} in source
// pixels, w = 0 when there is nothing to prefetch (exterior, ill-conditioned or non-finite tile).
VIDC_HD void fwd_tile_src_box(const vidc_frame_params& p, const vidc_camera& cam, int tx, int ty, uint32_t out[4]) {
    out[0] = out[1] = out[2] = out[3] = 0u;
    const float Wf = (float)cam.W, Hf = (float)cam.H;
    const float X[2] = {(float)(tx * 32), fminf((float)(tx * 32 + 31), Wf - 1.0f)};
    const float Y[2] = {(float)(ty * 32), fminf((float)(ty * 32 + 31), Hf - 1.0f)};
    float ix_lo = 3.0e38f, ix_hi = -3.0e38f, iy_lo = 3.0e38f, iy_hi = -3.0e38f, s_lo = 3.0e38f, s_hi = -3.0e38f;
    bool ok = true;
    for (int c = 0; c < 4; ++c) {
        const float px = p.ikw * X[c & 1] + p.px_min, py = p.ikh * Y[c >> 1] + p.py_min;
        const float t0 = p.Hinv[6] * px, t1 = p.Hinv[7] * py;
        const float s = t0 + t1 + p.Hinv[8];
        const float u = p.Hinv[0] * px + p.Hinv[1] * py + p.Hinv[2];
        const float v = p.Hinv[3] * px + p.Hinv[4] * py + p.Hinv[5];
        ok = ok && fabsf(s) > 1e-3f * (fabsf(t0) + fabsf(t1) + fabsf(p.Hinv[8]));
        const float ix = ((u / s - cam.cx) * cam.inv_half_w + 1.0f) * Wf * 0.5f - 0.5f;
        const float iy = ((v / s - cam.cy) * cam.inv_half_h + 1.0f) * Hf * 0.5f - 0.5f;
        ok = ok && fabsf(ix) < 1e8f && fabsf(iy) < 1e8f;
        ix_lo = fminf(ix_lo, ix); ix_hi = fmaxf(ix_hi, ix); iy_lo = fminf(iy_lo, iy); iy_hi = fmaxf(iy_hi, iy);
        s_lo = fminf(s_lo, s); s_hi = fmaxf(s_hi, s);
    }
    if (!(ok && (s_lo > 0.0f || s_hi < 0.0f))) return;
    int x0 = (int)floorf(ix_lo), x1 = (int)floorf(ix_hi) + 1, y0 = (int)floorf(iy_lo), y1 = (int)floorf(iy_hi) + 1;
    x0 = x0 < 0 ? 0 : x0; y0 = y0 < 0 ? 0 : y0;
    x1 = x1 > cam.W - 1 ? cam.W - 1 : x1; y1 = y1 > cam.H - 1 ? cam.H - 1 : y1;
    if (x1 < x0 || y1 < y0) return;
    out[0] = (uint32_t)x0; out[1] = (uint32_t)y0; out[2] = (uint32_t)(x1 - x0 + 1); out[3] = (uint32_t)(y1 - y0 + 1);
}

// ---- inverse warp: per-tile footprint boxes (kernels_box.cuh) -----------------------------------------------------------------
// The inverse warp of a 32x32 camera tile reads a canvas patch of about the same size.  unwarp_normals_box_kernel stages
// that patch in shared memory with coalesced 128-bit loads and takes its bilinear taps from there; which patch to stage is
// decided here, once per frame and tile, by the per-frame kernel.  NOT part of any result: a pixel whose taps do not lie
// inside the staged box takes the kernel's direct (global-memory) path, so a wrong box can only cost time.
//
// Entry layout (4 x uint32 per tile):
//   [0] box A: (x0 & 0xffff) | (y0 << 16)          [1] w | h << 8 | nsub << 16 | sigma << 20 | div_proven << 21
//   [2] box B: (x0 & 0xffff) | (y0 << 16)          [3] w | h << 8
// nsub = 1: box A covers the whole tile; 2: A covers tile rows 0..15 and B rows 16..31; 0: nothing is staged (pole inside the
// tile or a footprint that does not fit).  x0 is a multiple of 4 (it may be -4), the box includes the +1 taps and may overhang
// the image by up to 4 columns / 1 row (staged as zeros = padding_mode='zeros').  sigma selects the row pitch of the staging
// buffer (65 or 63 floats, i.e. +-1 modulo the 32 banks) so that the 32 taps of a canvas row segment fall into distinct banks.
#ifndef VIDC_BOX_MAX_H
#define VIDC_BOX_MAX_H 40
#endif
constexpr int kBoxMaxW = 60, kBoxMaxH = VIDC_BOX_MAX_H;        // 60: whole float4 groups (columns 56..59) stay inside a 63-float row pitch

struct InvBox { int x0, y0, w, h; bool ok; };

VIDC_HD void inv_pixel_coords(const vidc_frame_params& p, const vidc_camera& cam, float X, float Y, float& ix, float& iy, float& s_out,
                              float& s_terms) {
    const float* Hm = p.H;
    const float u = fmaf(Hm[1], Y, Hm[0] * X) + Hm[2];
    const float v = fmaf(Hm[4], Y, Hm[3] * X) + Hm[5];
    const float s = fmaf(Hm[7], Y, Hm[6] * X) + Hm[8];
    const float tx = u / s, ty = v / s;
    const float gx = cam.inv_half_w * (p.kw * (tx - p.px_min) - cam.cx);
    const float gy = cam.inv_half_h * (p.kh * (ty - p.py_min) - cam.cy);
    ix = fmaf(gx + 1.0f, (float)cam.W, -1.0f) * 0.5f;
    iy = fmaf(gy + 1.0f, (float)cam.H, -1.0f) * 0.5f;
    s_out = s;
    s_terms = fabsf(Hm[6] * X) + fabsf(Hm[7] * Y) + fabsf(Hm[8]);
}

// Bounding box of the taps of camera pixels [X0, X1] x [Y0, Y1] (inclusive).  Over a rectangle on which the projective
// denominator keeps its sign the map is continuous and takes the rectangle into the convex quadrilateral of its mapped
// corners, so the extremes of both coordinates are at the corners; 0.02 px absorbs the fp32 evaluation error.
VIDC_HD InvBox inv_rect_box(const vidc_frame_params& p, const vidc_camera& cam, int X0, int Y0, int X1, int Y1) {
    InvBox b; b.x0 = 0; b.y0 = 0; b.w = 1; b.h = 1; b.ok = false;
    float xlo = 3.0e38f, xhi = -3.0e38f, ylo = 3.0e38f, yhi = -3.0e38f, slo = 3.0e38f, shi = -3.0e38f;
    bool ok = true;
    for (int c = 0; c < 4; ++c) {
        float ix, iy, s, st;
        inv_pixel_coords(p, cam, (float)((c & 1) ? X1 : X0), (float)((c >> 1) ? Y1 : Y0), ix, iy, s, st);
        ok = ok && fabsf(s) > 1e-3f * st && fabsf(ix) < 1e8f && fabsf(iy) < 1e8f;       // also rejects NaN
        xlo = fminf(xlo, ix); xhi = fmaxf(xhi, ix); ylo = fminf(ylo, iy); yhi = fmaxf(yhi, iy);
        slo = fminf(slo, s); shi = fmaxf(shi, s);
    }
    ok = ok && (slo > 0.0f || shi < 0.0f);
    if (!ok) return b;
    int x_lo = (int)floorf(xlo - 0.02f), x_hi = (int)floorf(xhi + 0.02f) + 1;
    int y_lo = (int)floorf(ylo - 0.02f), y_hi = (int)floorf(yhi + 0.02f) + 1;
    x_lo = x_lo < -1 ? -1 : x_lo; y_lo = y_lo < -1 ? -1 : y_lo;
    x_hi = x_hi > cam.W ? cam.W : x_hi; y_hi = y_hi > cam.H ? cam.H : y_hi;
    if (x_hi <= x_lo || y_hi <= y_lo) { b.ok = true; return b; }          // maps outside the canvas: empty box, all zeros
    b.x0 = (x_lo >> 2) << 2;                                              // floor to a multiple of 4 (arithmetic shift)
    b.y0 = y_lo;
    b.w = x_hi - b.x0 + 1;
    b.h = y_hi - y_lo + 1;
    b.ok = b.w <= kBoxMaxW && b.h <= kBoxMaxH;
    if (!b.ok) { b.x0 = 0; b.y0 = 0; b.w = 1; b.h = 1; }
    return b;
}

// torchvision's ToTensor on a uint8 image (dataset.py:468-471: PIL image -> to_tensor): img.to(float32).div(255), one correctly
// rounded fp32 division per value.  q = x c with c = fl(1 / 255), r = x - 255 q (exact in one FMA), q + r c: the correctly
// rounded quotient for every x in 0..255 (all 256 values are compared with torch in tests/test_product_host_math.py).
VIDC_HD float u8_to_unit(unsigned int p) {
    const float x = (float)p, c = 0.003921568859368563f;
    const float q = x * c;
    const float r = fmaf(-q, 255.0f, x);
    return fmaf(r, c, q);
}

// The shared-reciprocal division of the hot kernels (kernels_fast.cuh: div2_rn) is the correctly rounded quotient while
// |s| lies in [2^-40, 2^40] and each numerator is zero or lies in [2^-80, 2^80].  For the inverse warp u, v, s are
// fma(H1, Y, H0 X) + H2 with integer pixel coordinates 0 <= X, Y < 2^15, so a non-zero numerator is a multiple of the
// smallest ulp among its non-zero coefficients: with every non-zero |H_k| in [2^-56, 2^60] it is >= 2^-80 and <= 2^80.
// s is affine in (X, Y): if its four image-corner values share a sign and exceed 2^-10 of M = |H6| W + |H7| H + |H8| (the
// rounding error of the evaluation is < 2^-21 M), then 2^-11 M <= |s| <= 1.01 M everywhere; M in [2^-25, 2^39] closes it.
// A frame that passes runs the inverse kernel WITHOUT the per-pixel window test (six instructions per pixel).
VIDC_HD bool inv_division_proven(const vidc_frame_params& p, const vidc_camera& cam) {
    const float* Hm = p.H;
    bool ok = cam.W <= 32768 && cam.H <= 32768;
    for (int k = 0; k < 9; ++k) {
        const float a = fabsf(Hm[k]);
        ok = ok && (a == 0.0f || (a >= 0x1p-56f && a <= 0x1p60f));        // NaN fails both
    }
    const float Wm = (float)(cam.W - 1), Hh = (float)(cam.H - 1);
    const float M = fabsf(Hm[6]) * (float)cam.W + fabsf(Hm[7]) * (float)cam.H + fabsf(Hm[8]);
    ok = ok && M >= 0x1p-25f && M <= 0x1p39f;
    float slo = 3.0e38f, shi = -3.0e38f;
    for (int c = 0; c < 4; ++c) {
        const float s = fmaf(Hm[7], (c >> 1) ? Hh : 0.0f, Hm[6] * ((c & 1) ? Wm : 0.0f)) + Hm[8];
        slo = fminf(slo, s); shi = fmaxf(shi, s);
    }
    const float m = slo > 0.0f ? slo : -shi;                              // smallest corner magnitude if the sign is common
    return ok && (slo > 0.0f || shi < 0.0f) && m >= 0x1p-10f * M;
}

// Canvas box of the inverse warp's L2 prefetch (kernels_shear.cuh: inv_prefetch_tile): out = {x0, y0, x1, y1} (inclusive,
// clipped to the canvas) holds both bilinear taps of every camera pixel of [X0, X1] x [Y0, Y1].  Only for frames that pass
// inv_division_proven: there s keeps its sign over the image, so (as in inv_rect_box) the mapped rectangle lies in the box of
// its mapped corners; the 2 px margin holds the +1 taps and the difference between this evaluation (one approximate
// reciprocal per corner) and the kernels' correctly rounded one.  A hint only.  false: nothing to prefetch (non-finite, or off the canvas).
VIDC_HD bool inv_prefetch_box(const float* Hm, float px_min, float py_min, float kw, float kh, float cx, float cy, float ihw,
                              float ihh, int W, int H, int X0, int Y0, int X1, int Y1, int out[4]) {
    float xlo = 3.0e38f, xhi = -3.0e38f, ylo = 3.0e38f, yhi = -3.0e38f;
#pragma unroll 1
    for (int c = 0; c < 4; ++c) {                                     // not unrolled: few live registers in the kernels' prologue
        const float X = (float)((c & 1) ? X1 : X0), Y = (float)((c >> 1) ? Y1 : Y0);
        const float u = fmaf(Hm[1], Y, Hm[0] * X) + Hm[2];
        const float v = fmaf(Hm[4], Y, Hm[3] * X) + Hm[5];
        const float s = fmaf(Hm[7], Y, Hm[6] * X) + Hm[8];
#ifdef __CUDA_ARCH__
        const float r = __fdividef(1.0f, s);                          // 2 ulp, and no slow-path call in the kernels' prologue
#else
        const float r = 1.0f / s;
#endif
        const float ix = fmaf(ihw * (kw * (u * r - px_min) - cx) + 1.0f, (float)W, -1.0f) * 0.5f;
        const float iy = fmaf(ihh * (kh * (v * r - py_min) - cy) + 1.0f, (float)H, -1.0f) * 0.5f;
        xlo = fminf(xlo, ix); xhi = fmaxf(xhi, ix); ylo = fminf(ylo, iy); yhi = fmaxf(yhi, iy);
    }
    if (!(xlo > -1.0e6f && xhi < 1.0e6f && ylo > -1.0e6f && yhi < 1.0e6f)) return false;       // also rejects NaN
    int x0 = (int)floorf(xlo) - 2, x1 = (int)floorf(xhi) + 3, y0 = (int)floorf(ylo) - 2, y1 = (int)floorf(yhi) + 3;
    x0 = x0 < 0 ? 0 : x0; y0 = y0 < 0 ? 0 : y0;
    x1 = x1 > W - 1 ? W - 1 : x1; y1 = y1 > H - 1 ? H - 1 : y1;
    out[0] = x0; out[1] = y0; out[2] = x1; out[3] = y1;
    return x0 <= x1 && y0 <= y1;
}

VIDC_HD void inv_tile_boxes(const vidc_frame_params& p, const vidc_camera& cam, int tx, int ty, bool div_proven, uint32_t out[4]) {
    const int X0 = tx * 32, Y0 = ty * 32;
    const int X1 = (X0 + 31 < cam.W - 1) ? X0 + 31 : cam.W - 1, Y1 = (Y0 + 31 < cam.H - 1) ? Y0 + 31 : cam.H - 1;
    // sigma: sign of d(canvas x)/dX * d(canvas y)/dX at the tile centre (kw, kh > 0 and the common 1/s^2 drop out)
    float ix, iy, s, st;
    const float Xc = (float)(X0 + 16), Yc = (float)(Y0 + 16);
    inv_pixel_coords(p, cam, Xc, Yc, ix, iy, s, st);
    const float u = fmaf(p.H[1], Yc, p.H[0] * Xc) + p.H[2], v = fmaf(p.H[4], Yc, p.H[3] * Xc) + p.H[5];
    const float dxdX = p.H[0] * s - u * p.H[6], dydX = p.H[3] * s - v * p.H[6];
    const uint32_t sigma = (dxdX * dydX >= 0.0f) ? 1u : 0u;
    InvBox a = inv_rect_box(p, cam, X0, Y0, X1, Y1), b2; b2.x0 = 0; b2.y0 = 0; b2.w = 1; b2.h = 1; b2.ok = false;
    uint32_t nsub = a.ok ? 1u : 0u;
    if (!a.ok && Y0 + 16 <= Y1) {
        const InvBox h0 = inv_rect_box(p, cam, X0, Y0, X1, Y0 + 15), h1 = inv_rect_box(p, cam, X0, Y0 + 16, X1, Y1);
        if (h0.ok && h1.ok) { a = h0; b2 = h1; nsub = 2u; }
    }
    out[0] = ((uint32_t)a.x0 & 0xffffu) | ((uint32_t)a.y0 << 16);
    out[1] = (uint32_t)a.w | ((uint32_t)a.h << 8) | (nsub << 16) | (sigma << 20) | ((div_proven ? 1u : 0u) << 21);
    out[2] = ((uint32_t)b2.x0 & 0xffffu) | ((uint32_t)b2.y0 << 16);
    out[3] = (uint32_t)b2.w | ((uint32_t)b2.h << 8);
}

}  // namespace vidc
