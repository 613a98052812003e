/*
 * backward_scatter.c -- the fixed summation order of vidc_warp_backward_ordered restated as a plain serial C loop.
 *
 * TEST INFRASTRUCTURE ONLY (tests/backward_oracle.py builds and loads it; the product never does).  The sampling grids and
 * the rotation R come from the CPU oracle (oracle/warp_oracle.c: vidc_oracle_forward_grid / vidc_oracle_inverse_grid /
 * vidc_oracle_build_homography), i.e. exactly the grids the warp methods sample with (no aspect guard).
 *
 * For each frame: every element of grad_in starts at +0; the output pixels are visited in row-major order (Y, then X) and
 * each adds, into each of its in-bounds taps, the product w_tap * g rounded and then added with a separate rounding (no FMA;
 * compile with -ffp-contract=off).  Bilinear taps nw, ne, sw, se with ATen's weights; nearest: the nearbyint tap, contribution
 * g itself.  A non-finite or out-of-int-range coordinate reads as -100 (GridSampler.cuh safe_downgrade_to_int_range): no tap
 * is in bounds.  R != NULL (inverse warp, C = 3): g <- R g first, k-ascending FMA chain from +0.
 */
#include <math.h>
#include <stddef.h>
#include <string.h>

#define API __attribute__((visibility("default")))

static inline float unnormalize(float g, int size) { return fmaf(g + 1.0f, (float)size, -1.0f) / 2.0f; }
static inline float safe_downgrade(float x)
{
    if (x > 2147483646.0f || x < -2147483648.0f || !isfinite(x)) return -100.0f;
    return x;
}

/* grad_out (B,C,H,W), grid (B,H,W,2), R (B,3,3) or NULL, grad_in (B,C,Hin,Win); all contiguous.  C <= 64. */
API void vidc_test_backward_scatter(const float *grad_out, int B, int C, int H, int W, const float *grid, const float *R,
                                    int Hin, int Win, int mode, float *grad_in)
{
    const size_t hw = (size_t)H * W, ihw = (size_t)Hin * Win;
    memset(grad_in, 0, sizeof(float) * ihw * (size_t)C * (size_t)B);
    float gv[64];
    for (int b = 0; b < B; ++b) {
        const float *gb = grad_out + (size_t)b * C * hw, *gr = grid + (size_t)b * hw * 2, *Rb = R ? R + 9 * b : NULL;
        float *ob = grad_in + (size_t)b * C * ihw;
        for (int Y = 0; Y < H; ++Y)
            for (int X = 0; X < W; ++X) {
                const size_t p = (size_t)Y * W + X;
                for (int c = 0; c < C; ++c) gv[c] = gb[c * hw + p];
                if (Rb) {                                  /* z = R^T y  =>  dL/dy = R dL/dz */
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
                        for (int c = 0; c < C; ++c) {
                            float *e = ob + c * ihw + (size_t)ty[t] * Win + tx[t];
                            const float prod = w[t] * gv[c];
                            *e = *e + prod;
                        }
                    }
                } else {
                    const int xn = (int)nearbyintf(ix), yn = (int)nearbyintf(iy);
                    if (xn < 0 || xn >= Win || yn < 0 || yn >= Hin) continue;
                    for (int c = 0; c < C; ++c) {
                        float *e = ob + c * ihw + (size_t)yn * Win + xn;
                        *e = *e + gv[c];
                    }
                }
            }
    }
}
