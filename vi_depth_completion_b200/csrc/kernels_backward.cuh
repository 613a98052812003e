// kernels_backward.cuh -- backward (scatter-add) kernels, row f4
// Part of libvidc_b200.so (one translation unit, vidc_kernels.cu); compiled with -fmad=false.
#pragma once
#include "device_common.cuh"

namespace vidc_k {

// ------------------------------------------------------------------------------------------
// Backward kernels (SURVEY.md section 8 row f4): gradient w.r.t. the sampled image.  Same coordinates as the
// forward kernels; each output-gradient pixel scatters w_tap * g into its (in-bounds) taps with atomicAdd, as
// ATen's grid_sampler_2d_backward does on CUDA.  The sum order is therefore not deterministic: each element S is an
// fp32 sum, from the memset's +0 in some order, of its k terms t, and tests/test_gpu_atomic_backward.py holds it to
// that: k = 0 gives +0, k <= 2 the order-free bits of (+0 + t1) + t2, NaN / infinite terms the IEEE result, and finite
// terms |S - E| <= gamma_{k-1} sum|t| + k 2^-52 sum|t| + k 2^-126 (E the exact sum, gamma_n = n u / (1 - n u),
// u = 2^-24); the last term because the fp32 atomicAdd flushes subnormal terms and sums to zero (measured on a B200).
// ROT: the incoming gradient is first rotated, g <- R g (the forward pass of the inverse warp applied R^T after
// sampling, :253).
template <bool INVERSE>
__global__ void __launch_bounds__(256)
warp_backward_kernel(const vidc_frame_params* __restrict__ prm, CamConst cam, ImgView gy /* (B,C,H,W) grad of the output */,
                     int C, int mode, float* __restrict__ gx, long long gx_sn, int gx_sc, int Hin, int Win) {
    const int b = blockIdx.z;
    const int X = blockIdx.x * blockDim.x + threadIdx.x;
    const int Y = blockIdx.y * blockDim.y + threadIdx.y;
    if (X >= cam.W || Y >= cam.H) return;
    const vidc_frame_params* __restrict__ P = prm + b;
    float M[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) M[k] = INVERSE ? __ldg(&P->H[k]) : __ldg(&P->Hinv[k]);
    const float px_min = __ldg(&P->px_min), py_min = __ldg(&P->py_min);
    float ix, iy;
    if (INVERSE) inverse_coords(M, px_min, py_min, __ldg(&P->kw), __ldg(&P->kh), cam, (float)X, (float)Y, (float)Win, (float)Hin, ix, iy);
    else forward_coords(M, px_min, py_min, __ldg(&P->ikw), __ldg(&P->ikh), cam, (float)X, (float)Y, (float)Win, (float)Hin, ix, iy);
    const float* __restrict__ g = gy.p + (long long)b * gy.sn + Y * gy.sh + X * gy.sw;
    float gv[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) gv[c] = c < C ? __ldg(g + c * gy.sc) : 0.0f;
    if (INVERSE) {   // z = R^T y  =>  dL/dy = R dL/dz
        float R[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) R[k] = __ldg(&P->R[k]);
        const float a0 = gv[0], a1 = gv[1], a2 = gv[2];
        gv[0] = fmaf(R[2], a2, fmaf(R[1], a1, fmaf(R[0], a0, 0.0f)));
        gv[1] = fmaf(R[5], a2, fmaf(R[4], a1, fmaf(R[3], a0, 0.0f)));
        gv[2] = fmaf(R[8], a2, fmaf(R[7], a1, fmaf(R[6], a0, 0.0f)));
    }
    float* __restrict__ out = gx + (long long)b * gx_sn;
    if (mode == VIDC_BILINEAR) {
        const Taps t = bilinear_taps(ix, iy, Hin, Win, Win, 1);
        for (int c = 0; c < C; ++c) {
            float* __restrict__ pl = out + (long long)c * gx_sc;
            if (t.b_nw) atomicAdd(pl + t.o_nw, t.w_nw * gv[c]);
            if (t.b_ne) atomicAdd(pl + t.o_ne, t.w_ne * gv[c]);
            if (t.b_sw) atomicAdd(pl + t.o_sw, t.w_sw * gv[c]);
            if (t.b_se) atomicAdd(pl + t.o_se, t.w_se * gv[c]);
        }
    } else {
        const int xn = (int)rintf(ix), yn = (int)rintf(iy);
        if ((unsigned)xn < (unsigned)Win && (unsigned)yn < (unsigned)Hin)
            for (int c = 0; c < C; ++c) atomicAdd(out + (long long)c * gx_sc + yn * Win + xn, gv[c]);
    }
}

}  // namespace vidc_k
