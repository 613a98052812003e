/*
 * exact_reference.c -- exact references for the outputs whose kernels are not pinned by a serial restatement:
 *   vidc_test_scatter_stats   per grad_in element, the terms the atomic image backward (vidc_warp_backward) adds: their count,
 *                             their exact (fp64) sum, the sum of their magnitudes, their special values and the order-free
 *                             result of one or two of them;
 *   vidc_test_touch_plane     the validity plane of the inverse warp (unwarp_normals(..., with_valid=True));
 *   vidc_test_rotate          z = R y of the rotated forward warp (warp_normal_image_with_gravity_center_aligned);
 *   vidc_test_homography_grid the sampling grid of warp_with_homography, from its fp32 frame parameters.
 *
 * TEST INFRASTRUCTURE ONLY (tests/exact_reference.py builds and loads it; the product never does).  The grids and R come from
 * the CPU oracle (oracle/warp_oracle.c), exactly as tests/harness/backward_scatter.c takes them.  Every fp32 operation is
 * separately rounded unless written as fmaf(); compile with -ffp-contract=off.
 */
#include <math.h>
#include <float.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#define API __attribute__((visibility("default")))

enum { F_NAN = 1, F_PINF = 2, F_NINF = 4, F_SUBNORMAL = 8 };

static inline float unnormalize(float g, int size) { return fmaf(g + 1.0f, (float)size, -1.0f) / 2.0f; }
static inline float safe_downgrade(float x)
{
    if (x > 2147483646.0f || x < -2147483648.0f || !isfinite(x)) return -100.0f;
    return x;
}
static inline int subnormal(float x) { return x != 0.0f && fabsf(x) < FLT_MIN; }

static inline void add_term(size_t e, float t, int32_t *k, double *E, double *A, uint8_t *flags, float *pair)
{
    const int32_t n = k[e]++;
    if (isnan(t)) flags[e] |= F_NAN;
    else if (isinf(t)) flags[e] |= t > 0 ? F_PINF : F_NINF;
    else { E[e] += (double)t; A[e] += fabs((double)t); }
    if (subnormal(t)) flags[e] |= F_SUBNORMAL;
    /* the atomic sum starts from the +0 of the memset; with one or two terms every order gives (+0 + t1) + t2 */
    if (n < 2) {
        pair[e] = pair[e] + t;
        if (n == 1 && subnormal(pair[e])) flags[e] |= F_SUBNORMAL;
    }
}

/* grad_out (B,C,H,W), grid (B,H,W,2), R (B,3,3) or NULL (inverse warp, C = 3: g <- R g first), outputs (B,C,Hin,Win); all
 * contiguous.  Terms as backward_scatter.c forms them: bilinear w_tap * g rounded once, nearest g itself. */
API void vidc_test_scatter_stats(const float *grad_out, int B, int C, int H, int W, const float *grid, const float *R, int Hin,
                                 int Win, int mode, int32_t *k, double *E, double *A, uint8_t *flags, float *pair)
{
    const size_t hw = (size_t)H * W, ihw = (size_t)Hin * Win, n = ihw * (size_t)C * (size_t)B;
    memset(k, 0, sizeof(int32_t) * n); memset(E, 0, sizeof(double) * n); memset(A, 0, sizeof(double) * n);
    memset(flags, 0, n); memset(pair, 0, sizeof(float) * n);
    float gv[64];
    for (int b = 0; b < B; ++b) {
        const float *gb = grad_out + (size_t)b * C * hw, *gr = grid + (size_t)b * hw * 2, *Rb = R ? R + 9 * b : NULL;
        const size_t ob = (size_t)b * C * ihw;
        for (size_t p = 0; p < hw; ++p) {
            for (int c = 0; c < C; ++c) gv[c] = gb[c * hw + p];
            if (Rb) {
                const float a0 = gv[0], a1 = gv[1], a2 = gv[2];
                gv[0] = fmaf(Rb[2], a2, fmaf(Rb[1], a1, fmaf(Rb[0], a0, 0.0f)));
                gv[1] = fmaf(Rb[5], a2, fmaf(Rb[4], a1, fmaf(Rb[3], a0, 0.0f)));
                gv[2] = fmaf(Rb[8], a2, fmaf(Rb[7], a1, fmaf(Rb[6], a0, 0.0f)));
            }
            const float ix = safe_downgrade(unnormalize(gr[2 * p], Win));
            const float iy = safe_downgrade(unnormalize(gr[2 * p + 1], Hin));
            if (mode == 0) {
                const float x0f = floorf(ix), y0f = floorf(iy);
                const int x0 = (int)x0f, y0 = (int)y0f;
                const float x1f = x0f + 1.0f, y1f = y0f + 1.0f;
                const float w[4] = {(x1f - ix) * (y1f - iy), (ix - x0f) * (y1f - iy), (x1f - ix) * (iy - y0f), (ix - x0f) * (iy - y0f)};
                const int tx[4] = {x0, x0 + 1, x0, x0 + 1}, ty[4] = {y0, y0, y0 + 1, y0 + 1};
                for (int t = 0; t < 4; ++t) {
                    if (tx[t] < 0 || tx[t] >= Win || ty[t] < 0 || ty[t] >= Hin) continue;
                    for (int c = 0; c < C; ++c)
                        add_term(ob + c * ihw + (size_t)ty[t] * Win + tx[t], w[t] * gv[c], k, E, A, flags, pair);
                }
            } else {
                const int xn = (int)nearbyintf(ix), yn = (int)nearbyintf(iy);
                if (xn < 0 || xn >= Win || yn < 0 || yn >= Hin) continue;
                for (int c = 0; c < C; ++c) add_term(ob + c * ihw + (size_t)yn * Win + xn, gv[c], k, E, A, flags, pair);
            }
        }
    }
}

/* grid (B,H,W,2) of the inverse warp -> touch (B,H,W): 1 where one of the four bilinear taps lies in [0,W)x[0,H), whatever
 * its weight (a tap at an exact-integer coordinate is in bounds with weight 0) */
API void vidc_test_touch_plane(const float *grid, int B, int H, int W, uint8_t *touch)
{
    const size_t hw = (size_t)H * W;
    for (size_t i = 0; i < hw * (size_t)B; ++i) {
        const float ix = safe_downgrade(unnormalize(grid[2 * i], W)), iy = safe_downgrade(unnormalize(grid[2 * i + 1], H));
        const int x0 = (int)floorf(ix), y0 = (int)floorf(iy);
        const int in_x = (x0 >= 0 && x0 < W) || (x0 + 1 >= 0 && x0 + 1 < W);
        const int in_y = (y0 >= 0 && y0 < H) || (y0 + 1 >= 0 && y0 + 1 < H);
        touch[i] = (uint8_t)(in_x && in_y);
    }
}

/* y (B,3,H,W) -> z = R y, z_c = fma(R[3c+2], y2, fma(R[3c+1], y1, fma(R[3c], y0, +0))) */
API void vidc_test_rotate(const float *y, int B, int H, int W, const float *R, float *z)
{
    const size_t hw = (size_t)H * W;
    for (int b = 0; b < B; ++b) {
        const float *Rb = R + 9 * b, *yb = y + 3 * hw * b;
        float *zb = z + 3 * hw * b;
        for (size_t p = 0; p < hw; ++p)
            for (int c = 0; c < 3; ++c)
                zb[c * hw + p] = fmaf(Rb[3 * c + 2], yb[2 * hw + p], fmaf(Rb[3 * c + 1], yb[hw + p], fmaf(Rb[3 * c], yb[p], 0.0f)));
    }
}

/* canvas (W,H) and the camera's cx, cy, inv_half_w, inv_half_h; per frame Hinv[9] and sc[4] = px_min, py_min, ikw, ikh (fp32)
 * -> grid (B,H,W,2): px = ikw X + px_min, u = fma(Hi1, py, Hi0 px) + Hi2, s likewise, sx = u / s, gx = inv_half_w (sx - cx) */
API void vidc_test_homography_grid(int W, int H, float cx, float cy, float inv_half_w, float inv_half_h, const float *Hinv,
                                   const float *sc, int B, float *grid)
{
    for (int b = 0; b < B; ++b) {
        const float *Hi = Hinv + 9 * b, *s4 = sc + 4 * b;
        float *gb = grid + (size_t)b * H * W * 2;
        for (int Y = 0; Y < H; ++Y)
            for (int X = 0; X < W; ++X) {
                const float px = s4[2] * (float)X + s4[0];
                const float py = s4[3] * (float)Y + s4[1];
                const float u = fmaf(Hi[1], py, Hi[0] * px) + Hi[2];
                const float v = fmaf(Hi[4], py, Hi[3] * px) + Hi[5];
                const float s = fmaf(Hi[7], py, Hi[6] * px) + Hi[8];
                const float sx = u / s, sy = v / s;
                float *o = gb + 2 * ((size_t)Y * W + X);
                o[0] = inv_half_w * (sx - cx);
                o[1] = inv_half_h * (sy - cy);
            }
    }
}
