// kernels_shear_cl.cuh -- the sheared warp kernels for CHANNELS-LAST three-channel images (torch.channels_last: pixel-
// interleaved, 12 bytes per pixel), for callers whose CNN runs in that memory format.
//
// Same segments, same arithmetic and therefore the same bits as kernels_shear.cuh; what changes is where a tap lives (the three
// channels of a pixel are adjacent: twelve 32-bit loads off one address, three per tap) and the shape of the staging tile: a
// row of the 32x32 tile is 96 consecutive floats of the output row, so the tile is the shared-memory image of a (96, 32) box of
// the output seen as a (3 W, H, B) tensor and leaves as ONE bulk tensor store.  A lane deposits at 3 * column + channel:
// 3 is coprime to the 32 banks, so deposits of lanes that run along X are conflict-free; tiles whose lanes run along Y
// (|roll| > 45 deg) take the same path with bank conflicts on their deposits (measured: tools/cl_time.py).
// Without these kernels channels-last tensors go through the strided kernels of kernels_generic.cuh (about half the speed).
#pragma once

namespace vidc_k {

struct ClStoreMaps {
    CUtensorMap img;                         // (3 W, H, B) fp32, box (96, 32, 1)
    CUtensorMap dep;                         // (W, H, B) fp32, box (32, 32, 1)
    CUtensorMap mask;                        // (W, H, B) uint8, box (32, 32, 1)
};

// bilinear taps of the three interleaved channels of one pixel position (row stride sh3 = 3 W floats)
__device__ __forceinline__ Px3 cl_sample_interior(const float* __restrict__ in, int sh3, const Pos& t) {
    Px3 o;
    const float* __restrict__ p = in + (t.y0 * sh3 + 3 * t.x0);
    o.a = bilerp(__ldg(p), __ldg(p + 3), __ldg(p + sh3), __ldg(p + sh3 + 3), t);
    o.b = bilerp(__ldg(p + 1), __ldg(p + 4), __ldg(p + sh3 + 1), __ldg(p + sh3 + 4), t);
    o.c = bilerp(__ldg(p + 2), __ldg(p + 5), __ldg(p + sh3 + 2), __ldg(p + sh3 + 5), t);
    return o;
}
__device__ __forceinline__ Px3 cl_sample_border(const float* __restrict__ in, int sh3, int Hin, int Win, const Pos& t) {
    const bool in_x0 = (unsigned)t.x0 < (unsigned)Win, in_x1 = (unsigned)(t.x0 + 1) < (unsigned)Win;
    const bool in_y0 = (unsigned)t.y0 < (unsigned)Hin, in_y1 = (unsigned)(t.y0 + 1) < (unsigned)Hin;
    const float* __restrict__ p0 = in + (t.y0 * sh3 + 3 * t.x0);
    const float* __restrict__ p1 = p0 + sh3;
    const bool nw = t.touch && in_x0 && in_y0, ne = t.touch && in_x1 && in_y0, sw = t.touch && in_x0 && in_y1, se = t.touch && in_x1 && in_y1;
    float v[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float v_nw = nw ? __ldg(p0 + c) : 0.0f, v_ne = ne ? __ldg(p0 + 3 + c) : 0.0f;
        const float v_sw = sw ? __ldg(p1 + c) : 0.0f, v_se = se ? __ldg(p1 + 3 + c) : 0.0f;
        v[c] = t.touch ? bilerp(v_nw, v_ne, v_sw, v_se, t) : 0.0f;         // as sample_border: a non-finite coordinate reads +0
    }
    Px3 o = {v[0], v[1], v[2]};
    return o;
}
__device__ __forceinline__ Px3 cl_sample(const float* __restrict__ in, int sh3, int H, int W, const Pos& t0) {
    Px3 o = {0.0f, 0.0f, 0.0f};
    if (__all_sync(0xffffffffu, t0.interior)) {
        o = cl_sample_interior(in, sh3, t0);
    } else {
        Pos t = t0;
        t.touch = t0.fin && (unsigned)(t0.x0 + 1) <= (unsigned)W && (unsigned)(t0.y0 + 1) <= (unsigned)H;
        if (__any_sync(0xffffffffu, t.touch)) o = cl_sample_border(in, sh3, H, W, t);
    }
    return o;
}

// ---- inverse: channels-last normals in, channels-last normals out ------------------------------------------------------------------
template <int GW, int GH, bool NORMALIZE, bool ALONG_Y>
__device__ __forceinline__ void unwarp_normals_cl_segments(const InvArgs& a, const float* pr, float (*tile)[96], int sh_l, bool proven) {
    const int W = GW ? GW : a.cam.W, H = GW ? GH : a.cam.H;
    const int b = blockIdx.z, lane = threadIdx.x, warp = threadIdx.y;
    const int tileX0 = blockIdx.x * TILE_W, tileY0 = blockIdx.y * TILE_H;
    const float* R = pr + 9;
    const float* __restrict__ in = a.x + (long long)b * a.x_sn;
    const InvShearChain<ALONG_Y> chain(pr, W, H, tileX0, tileY0, lane);
#pragma unroll
    for (int j = 0; j < ROWS_PER_THREAD; ++j) {
        const int S = (VIDC_SEG(warp, j) + sh_l) & 31;
        const Pos t = chain.at(S, proven, a.cam);
        const Px3 y = cl_sample(in, 3 * W, H, W, t);
        float z0 = fmaf(R[6], y.c, fmaf(R[3], y.b, fmaf(R[0], y.a, 0.0f)));    // :253
        float z1 = fmaf(R[7], y.c, fmaf(R[4], y.b, fmaf(R[1], y.a, 0.0f)));
        float z2 = fmaf(R[8], y.c, fmaf(R[5], y.b, fmaf(R[2], y.a, 0.0f)));
        if (NORMALIZE) normalize3_rn(z0, z1, z2);                  // surface_normal.py:170
        const int row = ALONG_Y ? lane : S, col = ALONG_Y ? S : lane;
        float* __restrict__ d = &tile[row][3 * col];
        d[0] = z0; d[1] = z1; d[2] = z2;
    }
}

template <int GW, int GH, bool NORMALIZE>
__global__ void __launch_bounds__(256, GW ? VIDC_SHEAR_BLOCKS_INV : VIDC_SHEAR_BLOCKS_RT)
unwarp_normals_shear_cl_kernel(const __grid_constant__ InvArgs a, const __grid_constant__ ClStoreMaps maps) {
    static_assert(GW % 32 == 0, "sheared tiles need a canvas whose width is a multiple of 32 (GW = 0: runtime geometry)");
    __shared__ __align__(128) float tile[32][96];
    const int b = blockIdx.z, lane = threadIdx.x, warp = threadIdx.y;
    const int tileX0 = blockIdx.x * TILE_W, tileY0 = blockIdx.y * TILE_H;
    float pr[32];
    load_params(a.prm + b, pr, 0, 8);
    int sh_l;
    const bool along_y = inv_shear_of_tile(pr, tileX0, tileY0, lane, sh_l);
    const bool proven = __ldg(&a.prm[b].reserved[10]) != 0.0f;     // CTA-uniform (vidc::inv_division_proven)
    if (along_y) unwarp_normals_cl_segments<GW, GH, NORMALIZE, true>(a, pr, tile, sh_l, proven);
    else unwarp_normals_cl_segments<GW, GH, NORMALIZE, false>(a, pr, tile, sh_l, proven);
    fence_async_smem();
    __syncthreads();
    if (warp == 0 && lane == 0) {
        tma_store_3d(&maps.img, &tile[0][0], 3 * tileX0, tileY0, b);
        tma_store_commit_and_wait_read();
    }
}

// ---- forward: channels-last RGB in / out, planar depth (one channel is the same in both formats), mask, coverage --------------------
template <int GW, int GH, bool HAS_D, bool ALONG_Y>
__device__ __forceinline__ unsigned int warp_rgbd_cl_segments(const FwdArgs& a, const float* pr, float (*tile)[96], float (*dtile)[32],
                                                              unsigned char (*mt)[32], int sh_l) {
    const int W = GW ? GW : a.cam.W, H = GW ? GH : a.cam.H;
    const int b = blockIdx.z, lane = threadIdx.x, warp = threadIdx.y;
    const int tileX0 = blockIdx.x * TILE_W, tileY0 = blockIdx.y * TILE_H;
    const float* __restrict__ in_rgb = a.rgb + (long long)b * a.rgb_sn;
    const float* __restrict__ in_dep = HAS_D ? a.dep + (long long)b * a.dep_sn : nullptr;
    const FwdShearChain<ALONG_Y> chain(pr, W, H, tileX0, tileY0, lane);
    unsigned int cnt = 0;
#pragma unroll
    for (int j = 0; j < ROWS_PER_THREAD; ++j) {
        const int S = (VIDC_SEG(warp, j) + sh_l) & 31;
        float ix, iy;
        const Pos t = chain.at(S, a.cam, ix, iy);
        Px3 o = {0.0f, 0.0f, 0.0f};
        float od = 0.0f;
        if (__any_sync(0xffffffffu, t.touch)) {                    // exterior segments: zeros
            if (__all_sync(0xffffffffu, t.interior)) {
                o = cl_sample_interior(in_rgb, 3 * W, t);
                if (HAS_D) od = a.mode_d == VIDC_BILINEAR ? sample_interior(in_dep, t.y0 * W + t.x0, W, t) : sample_nearest_pos(in_dep, ix, iy, H, W, W, true);
            } else {
                o = cl_sample_border(in_rgb, 3 * W, H, W, t);
                if (HAS_D) od = a.mode_d == VIDC_BILINEAR ? sample_border(in_dep, W, H, W, t) : sample_nearest_pos(in_dep, ix, iy, H, W, W, t.touch);
            }
        }
        const int row = ALONG_Y ? lane : S, col = ALONG_Y ? S : lane;
        float* __restrict__ d = &tile[row][3 * col];
        d[0] = o.a; d[1] = o.b; d[2] = o.c;
        if (HAS_D) dtile[row][col] = od;
        if (a.mask || a.coverage) {                                // surface_normal.py:151
            const unsigned int m = (o.a + o.b) + o.c > 0.01f;
            mt[row][col] = (unsigned char)m;
            if ((GW && GH % 32 == 0) || tileY0 + row < H) cnt += m;
        }
    }
    return cnt;
}

template <int GW, int GH, bool HAS_D>
__global__ void __launch_bounds__(256, GW ? VIDC_SHEAR_BLOCKS_FWD : VIDC_SHEAR_BLOCKS_RT)
warp_rgbd_shear_cl_kernel(const __grid_constant__ FwdArgs a, const __grid_constant__ ClStoreMaps maps) {
    static_assert(GW % 32 == 0, "sheared tiles need a canvas whose width is a multiple of 32 (GW = 0: runtime geometry)");
    __shared__ __align__(128) float tile[32][96];
    __shared__ __align__(128) float dtile[HAS_D ? 32 : 1][32];
    __shared__ __align__(128) unsigned char mtile[32][32];
    const int b = blockIdx.z, lane = threadIdx.x, warp = threadIdx.y;
    const int tileX0 = blockIdx.x * TILE_W, tileY0 = blockIdx.y * TILE_H;
    float pr[20];
    load_params(a.prm + b, pr, 4, 5);
    int sh_l;
    const bool along_y = fwd_shear_of_tile(pr, tileX0, tileY0, lane, sh_l);
    // (the exterior-tile bitmap is not consulted here: exterior segments already cost one vote and three zero deposits)
    unsigned int cnt = along_y ? warp_rgbd_cl_segments<GW, GH, HAS_D, true>(a, pr, tile, dtile, mtile, sh_l)
                               : warp_rgbd_cl_segments<GW, GH, HAS_D, false>(a, pr, tile, dtile, mtile, sh_l);
    fence_async_smem();
    __syncthreads();
    if (warp == 0 && lane == 0) {
        tma_store_3d(&maps.img, &tile[0][0], 3 * tileX0, tileY0, b);
        if (HAS_D) tma_store_3d(&maps.dep, &dtile[0][0], tileX0, tileY0, b);
        if (a.mask) tma_store_3d(&maps.mask, &mtile[0][0], tileX0, tileY0, b);
        tma_store_commit_and_wait_read();
    }
    if (a.coverage) {
        cnt = __reduce_add_sync(0xffffffffu, cnt);
        if (lane == 0 && cnt) atomicAdd(a.coverage + b, cnt);
    }
}

}  // namespace vidc_k
