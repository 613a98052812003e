// vidc_kernels.cu -- the single translation unit of libvidc_b200.so: host-side dispatch and the C ABI
// (include/vidc_b200.h) of the gravity warp / unwarp path.  Compile with -fmad=false: the fp32 roundings in the
// kernels are the reference's.
//
//   exact_math.cuh / frame_params.cuh   bit-exact per-frame arithmetic (__host__ __device__, also built by the tests)
//   device_common.cuh                   image views, ATen grid_sampler primitives, the exact coordinate chains
//   kernels_params.cuh                  frame parameters (:35-58, :125-140), gravity conditioning, rasterisation
//   kernels_generic.cuh                 any-stride forward / inverse kernels, sampler grids (:158-214), masks, statistics
//   kernels_fast.cuh                    straight-row warp kernels (planar NCHW), incl. the column-major tile path: fallbacks
//   kernels_packed.cuh                  packed RGBD (channels-last C=4) forward kernel
//   kernels_shear.cuh                   THE SHIPPING WARP KERNELS: sheared segments (lanes follow source rows), L2 prefetch of a
//                                       later tile's source box, TMA write-out (bulk tensor stores from a planar staging tile)
//   kernels_shear_cl.cuh                the same for channels-last three-channel images (12-byte pixels, (96, 32) staging tile)
//   kernels_box.cuh                     inverse warp with the footprint staged in shared memory (opt-in, VIDC_INV_BOX=1)
//   kernels_backward.cuh                scatter-add backward
//   kernels_backward_ordered.cuh        gather backward in one fixed summation order (deterministic)
//   kernels_sparse.cuh                  sparse depth warped analytically (row f2)
//   tma_stage.cuh                       TMA / mbarrier PTX wrappers (bulk tensor loads and stores)
//   kernels_tma.cuh                     opt-in TMA-staged LOAD variants (VIDC_TMA=1)
#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <mutex>
#include <vector>

#include "frame_params.cuh"
#include "tma_stage.cuh"

#include "kernels_params.cuh"
#include "kernels_generic.cuh"
#include "kernels_fast.cuh"
#include "kernels_box.cuh"
#include "kernels_shear.cuh"
#include "kernels_shear_cl.cuh"
#include "kernels_backward.cuh"
#include "kernels_backward_ordered.cuh"
#include "kernels_sparse.cuh"
#include "kernels_packed.cuh"
#include "kernels_tma.cuh"

namespace vidc_k {


thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define VIDC_CUDA(expr)                                                                         \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return fail(VIDC_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(e_));         \
    } while (0)

#define VIDC_LAUNCH_CHECK()                                                                     \
    do {                                                                                        \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                     \
        cudaError_t e_ = cudaGetLastError();                                                    \
        if (e_ != cudaSuccess)                                                                  \
            return fail(VIDC_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e_));     \
    } while (0)

// self-test hook: the shared-reciprocal divisions against the compiler's IEEE division
__global__ void debug_div_kernel(const float* __restrict__ u, const float* __restrict__ v, const float* __restrict__ s,
                                 long long n, float* __restrict__ out /* [4][n]: fast u/s, fast v/s via div3, ref u/s, ref v/s */) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float qu, qv;
    div2_rn(u[i], v[i], s[i], qu, qv);
    float a = u[i], b = v[i], c = u[i];
    div3_rn(a, b, c, s[i]);
    out[i] = qu;
    out[n + i] = b;
    out[2 * n + i] = __fdiv_rn(u[i], s[i]);
    out[3 * n + i] = __fdiv_rn(v[i], s[i]);
    if (qv != b && !(qv != qv && b != b)) out[n + i] = __int_as_float(0x7fc00001);   // div2 and div3 must agree
}

// ------------------------------------------------------------------------------------------
// host helpers
int check_image(const vidc_image* im, const char* name, int want_c_min, int want_c_max) {
    if (!im) return fail(VIDC_ERR_INVALID_ARGUMENT, "%s: null image descriptor", name);
    if (!im->data && (long long)im->n * im->c * im->h * im->w != 0)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "%s: null data pointer", name);
    if (im->n < 0 || im->c < want_c_min || im->c > want_c_max || im->h < 0 || im->w < 0)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "%s: bad shape (%d,%d,%d,%d), channels must be in [%d,%d]", name,
                    im->n, im->c, im->h, im->w, want_c_min, want_c_max);
    if (im->n > 65535)   // frames ride on gridDim.z
        return fail(VIDC_ERR_INVALID_ARGUMENT, "%s: %d frames in one call, the limit is 65535 -- split the batch", name, im->n);
    const long long span = (long long)(im->c - 1) * im->sc + (long long)(im->h - 1) * im->sh + (long long)(im->w - 1) * im->sw;
    if (im->sc < 0 || im->sh < 0 || im->sw < 0 || im->sn < 0 || span >= (1LL << 31))
        return fail(VIDC_ERR_INVALID_ARGUMENT, "%s: strides must be non-negative and one frame must span < 2^31 elements", name);
    return VIDC_OK;
}
ImgView view_in(const vidc_image* im) {
    ImgView v; v.p = im->data; v.c = im->c; v.h = im->h; v.w = im->w; v.sn = im->sn;
    v.sc = (int)im->sc; v.sh = (int)im->sh; v.sw = (int)im->sw; return v;
}
ImgViewOut view_out(const vidc_image* im) {
    ImgViewOut v; v.p = im->data; v.c = im->c; v.h = im->h; v.w = im->w; v.sn = im->sn;
    v.sc = (int)im->sc; v.sh = (int)im->sh; v.sw = (int)im->sw; return v;
}
CamConst cam_const(const vidc_camera* cam) {
    CamConst c; c.cx = cam->cx; c.cy = cam->cy; c.inv_half_w = cam->inv_half_w; c.inv_half_h = cam->inv_half_h;
    c.W = cam->W; c.H = cam->H; return c;
}
int check_cam(const vidc_camera* cam) {
    if (!cam) return fail(VIDC_ERR_INVALID_ARGUMENT, "null camera");
    if (cam->W <= 0 || cam->H <= 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "camera has non-positive size %dx%d", cam->W, cam->H);
    return VIDC_OK;
}
dim3 grid2d(int W, int H, int B, dim3 blk) { return dim3((W + blk.x - 1) / blk.x, (H + blk.y - 1) / blk.y, B); }

int launch_params(const vidc_camera* cam, const float* d_Ig, const float* d_Ia, int B, vidc_frame_params* d_params,
                  cudaStream_t st, float* d_H_out = nullptr) {
    if (B == 0) return VIDC_OK;
    if (!d_Ig || !d_Ia || !d_params) return fail(VIDC_ERR_INVALID_ARGUMENT, "null gravity / alignment / params pointer");
    frame_params_kernel<<<(B + 63) / 64, 64, 0, st>>>(*cam, d_Ig, d_Ia, B, d_params, d_H_out);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}
// Parameters + exterior-tile bitmap for the sheared forward kernels (one CTA per frame); VIDC_TILE_SKIP=0 turns it off.
bool tile_skip_enabled() {
    static const bool v = [] { const char* e = getenv("VIDC_TILE_SKIP"); return !(e && e[0] == '0'); }();
    return v;
}
// L2 prefetch distance of the sheared forward kernel, in percent of a wave of resident CTAs (VIDC_FWD_PF_WAVES_X100, 0 = off).
// Measured (profiles/r2_history.md): 0.5605 ms without, 0.516-0.518 ms at 1-12 %, 0.538 at 50 %, 0.60 at a full wave.
int fwd_prefetch_pct() {
    static const int v = [] { const char* e = getenv("VIDC_FWD_PF_WAVES_X100"); return e ? atoi(e) : 8; }();
    return v;
}
int launch_params_tiles(const vidc_camera* cam, const float* d_Ig, const float* d_Ia, int B, vidc_frame_params* d_params,
                        cudaStream_t st, float* d_H_out) {
    if (B == 0) return VIDC_OK;
    if (!d_Ig || !d_Ia || !d_params) return fail(VIDC_ERR_INVALID_ARGUMENT, "null gravity / alignment / params pointer");
    static_assert(sizeof(vidc_frame_params) == 48 * sizeof(float), "frame params layout");
    // per-tile source boxes (prefetch hints) go behind the B parameter blocks of the caller's workspace (vidc_workspace_bytes)
    uint4* src_boxes = fwd_prefetch_pct() > 0 ? reinterpret_cast<uint4*>(d_params + B) : nullptr;
    frame_params_tiles_kernel<<<B, 320, 0, st>>>(*cam, d_Ig, d_Ia, B, d_params, d_H_out, src_boxes);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

// d_Ig == d_Ia == NULL: the workspace was prepared by vidc_frame_params_prepare (no per-frame kernel; Cg_H_C by a scatter if asked for)
int prepared_params(const vidc_frame_params* d_params_ws, int B, float* d_H_out, cudaStream_t st) {
    if (!d_params_ws) return fail(VIDC_ERR_INVALID_ARGUMENT, "null params pointer");
    if (d_H_out) {
        scatter_homography_kernel<<<(B * 9 + 127) / 128, 128, 0, st>>>(d_params_ws, B, d_H_out, nullptr, nullptr, nullptr);
        VIDC_LAUNCH_CHECK();
    }
    return VIDC_OK;
}

template <int C_A, bool HAS_D, bool ROT>
int launch_forward(const vidc_camera* cam, const vidc_frame_params* prm, const vidc_image* a, const vidc_image* ya, int mode_a,
                   const vidc_image* d, const vidc_image* yd, int mode_d, uint8_t* mask, uint32_t* cov, cudaStream_t st) {
    const dim3 blk(32, 8);
    ImgView dv{}; ImgViewOut ydv{};
    if (HAS_D) { dv = view_in(d); ydv = view_out(yd); }
    warp_forward_kernel<C_A, HAS_D, ROT><<<grid2d(cam->W, cam->H, a->n, blk), blk, 0, st>>>(
        prm, cam_const(cam), view_in(a), view_out(ya), mode_a, dv, ydv, mode_d, mask, cov);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int check_out(const vidc_camera* cam, const vidc_image* x, const vidc_image* y, const char* name) {
    if (y->n != x->n || y->c != x->c || y->h != cam->H || y->w != cam->W)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "%s: output must be (%d,%d,%d,%d), got (%d,%d,%d,%d)", name, x->n, x->c,
                    cam->H, cam->W, y->n, y->c, y->h, y->w);
    return VIDC_OK;
}

int scatter_h(const vidc_frame_params* prm, int B, float* H, float* R, float* Hi, float* Rt, cudaStream_t st) {
    if (B == 0 || (!H && !R && !Hi && !Rt)) return VIDC_OK;
    scatter_homography_kernel<<<(B * 9 + 127) / 128, 128, 0, st>>>(prm, B, H, R, Hi, Rt);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

// ---- TMA tensor maps (driver entry point resolved through the runtime, no libcuda link) -------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_encodeTiled tma_encoder() {
    static PFN_encodeTiled fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (PFN_encodeTiled)p;
    }();
    return fn;
}
// (W, H, C, N) fp32 view with a (64, box_h, C, 1) box; zero fill out of range.  false if the view cannot be described.
bool encode_image_map(CUtensorMap* map, const vidc_image* im, int box_h, int box_w = TMA_BW) {
    PFN_encodeTiled enc = tma_encoder();
    if (!enc || im->sw != 1) return false;
    if (((uintptr_t)im->data & 15) || (im->sh & 3) || (im->sc & 3) || (im->sn & 3) || im->sh <= 0 || im->sc <= 0) return false;
    if (im->w < 1 || im->h < 1) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)im->w, (cuuint64_t)im->h, (cuuint64_t)im->c, (cuuint64_t)im->n};
    const cuuint64_t strides[3] = {(cuuint64_t)im->sh * 4, (cuuint64_t)im->sc * 4, (cuuint64_t)(im->sn > 0 ? im->sn : im->sc * im->c) * 4};
    const cuuint32_t box[4] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)im->c, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, im->data, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// Output tensor maps of the TMA write-out (kernels_shear.cuh: StoreMaps): (W, H, C, N) fp32 planes, box (32, 32, C, 1), or
// (W, H, N) for a single plane.  false if the view cannot be described (strides not multiples of 16 bytes, ...).
bool encode_store_map(CUtensorMap* map, float* data, int W, int H, int C, int N, int64_t sh, int64_t sc, int64_t sn, bool plane3d = false) {
    PFN_encodeTiled enc = tma_encoder();
    if (!enc || ((uintptr_t)data & 15) || (sh & 3) || (sc & 3) || (sn & 3) || sh <= 0 || sn <= 0) return false;
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    if (plane3d) {                                   // StoreMaps::dep: one plane per frame, stored with the 3-D instruction
        const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
        const cuuint64_t strides[2] = {(cuuint64_t)sh * 4, (cuuint64_t)sn * 4};
        const cuuint32_t box[3] = {32, 32, 1};
        return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, data, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    }
    if (sc <= 0) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)N};
    const cuuint64_t strides[3] = {(cuuint64_t)sh * 4, (cuuint64_t)sc * 4, (cuuint64_t)sn * 4};
    const cuuint32_t box[4] = {32, 32, (cuuint32_t)C, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, data, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// channels-last three-channel image (kernels_shear_cl.cuh): the output seen as (3 W, H, N) fp32, box (96, 32, 1)
bool is_channels_last3(const vidc_image* im, int W, int H) {
    return im->c == 3 && im->w == W && im->h == H && im->sc == 1 && im->sw == 3 && im->sh == 3 * (int64_t)W && im->sn == 3 * (int64_t)W * H;
}
bool encode_cl_map(CUtensorMap* map, float* data, int W, int H, int N) {
    PFN_encodeTiled enc = tma_encoder();
    if (!enc || ((uintptr_t)data & 15) || (W & 3)) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)3 * W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t strides[2] = {(cuuint64_t)3 * W * 4, (cuuint64_t)3 * W * H * 4};
    const cuuint32_t box[3] = {96, 32, 1}, estr[3] = {1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, data, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
bool encode_mask_map(CUtensorMap* map, uint8_t* data, int W, int H, int N) {            // (W, H, N) uint8, contiguous, box (32, 32, 1)
    PFN_encodeTiled enc = tma_encoder();
    if (!enc || ((uintptr_t)data & 15) || (W & 15)) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
    const cuuint64_t strides[2] = {(cuuint64_t)W, (cuuint64_t)W * H};
    const cuuint32_t box[3] = {32, 32, 1}, estr[3] = {1, 1, 1};
    if (strides[1] & 15) return false;
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, data, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// TMA write-out of the sheared kernels (kernels_shear.cuh, StoreMaps): on unless VIDC_TMA_STORE=0 (A/B runs and the parity
// suite's handle on the LSU write-out); calls whose outputs cannot be described by a tensor map take the LSU write-out.
bool tma_store_enabled() {
    static const bool v = [] { const char* e = getenv("VIDC_TMA_STORE"); return !(e && e[0] == '0'); }();
    return v;
}
// The TMA-staged forward kernel is correct (parity suite) but, in its first one-tile-per-CTA form, slower than
// the L1-gather kernel on the B200 (0.89 vs 0.63 ms: exposed copy latency and 3-6x bounding-box over-fetch,
// profiles/r1_history.md), so it is opt-in: VIDC_TMA=1.
bool tma_enabled() {
    static const bool v = [] { const char* e = getenv("VIDC_TMA"); return e && e[0] == '1'; }();
    return v;
}

// Sheared row segments (kernels_shear.cuh).  VIDC_SHEAR = 2 (default): sheared forward and inverse warps; 1: sheared
// forward warp only; 0: straight rows everywhere.  Measured on the B200 the sheared kernels are at least as fast as the
// straight-row ones at every roll angle and 18-30 % faster beyond ~25 deg (profiles/r1_history.md); the switch exists
// for A/B measurements and as the parity suite's handle on each kernel family.
int shear_level() {
    static const int v = [] { const char* e = getenv("VIDC_SHEAR"); return (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 2; }();
    return v;
}
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// Inverse warp with the footprint staged in shared memory (kernels_box.cuh), for contiguous planes with W % 4 == 0.  Measured
// on the B200 it does not beat the sheared kernel (0.527 vs 0.499 ms, profiles/r2_history.md: the staging pass costs what the
// cheaper taps save), so it is opt-in: VIDC_INV_BOX=1 (A/B runs, and the parity suite's handle on it).
bool inv_box_enabled() {
    static const bool v = [] { const char* e = getenv("VIDC_INV_BOX"); return e && e[0] == '1'; }();
    return v;
}
template <typename K>
void prefer_shared_carveout(K kernel) {          // per device: function attributes belong to the device's context
    static std::atomic<unsigned long long> done[2] = {{0ull}, {0ull}};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 128) return;
    const unsigned long long bit = 1ull << (dev & 63);
    if (done[dev >> 6].load(std::memory_order_relaxed) & bit) return;
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    done[dev >> 6].fetch_or(bit, std::memory_order_relaxed);
}
template <int GW, int GH>
void launch_unwarp_box(bool normalize, bool has_valid, dim3 grd, dim3 blk, cudaStream_t st, const InvArgs& ia, const uint4* boxes) {
    const dim3 grd2(grd.x, (grd.y + 1) / 2, grd.z);               // one CTA = two vertically adjacent tiles
    // prefetch distance: about one wave of resident CTAs (SMs x CTAs per SM), as an offset in grid coordinates
    static const int wave = [] {
        int dev = 0, sms = 148;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const char* e = getenv("VIDC_BOX_PF_WAVES_X100");
        const int pct = e ? atoi(e) : 50;             // half a wave ahead measured best (0.527 ms; none 0.544, a full wave 0.63)
        return (int)((long long)sms * VIDC_BOX_BLOCKS * pct / 100);
    }();
    int3 pf;
    pf.x = wave % (int)grd2.x; pf.y = (wave / (int)grd2.x) % (int)grd2.y; pf.z = wave / (int)(grd2.x * grd2.y);
#define VIDC_BOX_LAUNCH(N, V)                                                          \
    do {                                                                               \
        prefer_shared_carveout(unwarp_normals_box_kernel<GW, GH, N, V>);               \
        unwarp_normals_box_kernel<GW, GH, N, V><<<grd2, blk, 0, st>>>(ia, boxes, (int)grd.y, pf); \
    } while (0)
    if (normalize) { if (has_valid) VIDC_BOX_LAUNCH(true, true); else VIDC_BOX_LAUNCH(true, false); }
    else { if (has_valid) VIDC_BOX_LAUNCH(false, true); else VIDC_BOX_LAUNCH(false, false); }
#undef VIDC_BOX_LAUNCH
}

template <int GW, int GH>
void launch_unwarp_shear(bool normalize, bool has_valid, bool ts, dim3 grd, dim3 blk, cudaStream_t st, const InvArgs& ia, const StoreMaps& sm) {
    if (ts && !has_valid) {
        if (normalize) unwarp_normals_shear_kernel<GW, GH, true, false, true><<<grd, blk, 0, st>>>(ia, sm);
        else unwarp_normals_shear_kernel<GW, GH, false, false, true><<<grd, blk, 0, st>>>(ia, sm);
    } else if (normalize) {
        if (has_valid) unwarp_normals_shear_kernel<GW, GH, true, true, false><<<grd, blk, 0, st>>>(ia, sm);
        else unwarp_normals_shear_kernel<GW, GH, true, false, false><<<grd, blk, 0, st>>>(ia, sm);
    } else {
        if (has_valid) unwarp_normals_shear_kernel<GW, GH, false, true, false><<<grd, blk, 0, st>>>(ia, sm);
        else unwarp_normals_shear_kernel<GW, GH, false, false, false><<<grd, blk, 0, st>>>(ia, sm);
    }
}
template <int GW, int GH>
void launch_rgbd_shear(bool has_d, bool ts, dim3 grd, dim3 blk, cudaStream_t st, const FwdArgs& fa, const StoreMaps& sm) {
    if (ts) {
        if (has_d) warp_rgbd_shear_kernel<GW, GH, true, true><<<grd, blk, 0, st>>>(fa, sm);
        else warp_rgbd_shear_kernel<GW, GH, false, true><<<grd, blk, 0, st>>>(fa, sm);
    } else {
        if (has_d) warp_rgbd_shear_kernel<GW, GH, true, false><<<grd, blk, 0, st>>>(fa, sm);
        else warp_rgbd_shear_kernel<GW, GH, false, false><<<grd, blk, 0, st>>>(fa, sm);
    }
}
template <int GW, int GH>
void launch_planes_shear(int C, bool ts, dim3 grd, dim3 blk, cudaStream_t st, const PlanesArgs& pa, const StoreMaps& sm) {
    if (ts) {
        if (C == 3) warp_planes_shear_kernel<GW, GH, 3, true><<<grd, blk, 0, st>>>(pa, sm);
        else warp_planes_shear_kernel<GW, GH, 1, true><<<grd, blk, 0, st>>>(pa, sm);
    } else {
        if (C == 3) warp_planes_shear_kernel<GW, GH, 3, false><<<grd, blk, 0, st>>>(pa, sm);
        else warp_planes_shear_kernel<GW, GH, 1, false><<<grd, blk, 0, st>>>(pa, sm);
    }
}

template <bool HAS_D>
void launch_rgbd_cl(const vidc_camera* cam, dim3 grd, dim3 blk, cudaStream_t st, const FwdArgs& fa, const ClStoreMaps& sm) {
    if (cam->W == 640 && cam->H == 480) warp_rgbd_shear_cl_kernel<640, 480, HAS_D><<<grd, blk, 0, st>>>(fa, sm);
    else if (cam->W == 320 && cam->H == 240) warp_rgbd_shear_cl_kernel<320, 240, HAS_D><<<grd, blk, 0, st>>>(fa, sm);
    else warp_rgbd_shear_cl_kernel<0, 0, HAS_D><<<grd, blk, 0, st>>>(fa, sm);
}
template <bool NORMALIZE>
void launch_unwarp_cl(const vidc_camera* cam, dim3 grd, dim3 blk, cudaStream_t st, const InvArgs& ia, const ClStoreMaps& sm) {
    if (cam->W == 640 && cam->H == 480) unwarp_normals_shear_cl_kernel<640, 480, NORMALIZE><<<grd, blk, 0, st>>>(ia, sm);
    else if (cam->W == 320 && cam->H == 240) unwarp_normals_shear_cl_kernel<320, 240, NORMALIZE><<<grd, blk, 0, st>>>(ia, sm);
    else unwarp_normals_shear_cl_kernel<0, 0, NORMALIZE><<<grd, blk, 0, st>>>(ia, sm);
}
// channels-last RGB (+ planar depth, mask, coverage) through warp_rgbd_shear_cl_kernel; false: not applicable, take another path
bool try_rgbd_cl(const vidc_camera* cam, const vidc_frame_params* prm, const vidc_image* rgb, const vidc_image* depth, int depth_mode,
                 const vidc_image* rgb_out, const vidc_image* depth_out, uint8_t* d_mask_u8, uint32_t* d_coverage, cudaStream_t st) {
    if (!(shear_level() >= 1 && tma_store_enabled() && cam->W % 32 == 0 && is_channels_last3(rgb, cam->W, cam->H) &&
          is_channels_last3(rgb_out, cam->W, cam->H))) return false;
    if (depth && !(depth->sw == 1 && depth->sh == cam->W && depth->w == cam->W && depth->h == cam->H && depth_out->sw == 1 && depth_out->sh == cam->W))
        return false;
    ClStoreMaps sm;
    if (!encode_cl_map(&sm.img, rgb_out->data, cam->W, cam->H, rgb->n)) return false;
    if (depth && !encode_store_map(&sm.dep, depth_out->data, cam->W, cam->H, 1, rgb->n, depth_out->sh, (int64_t)cam->W * cam->H, depth_out->sn, true)) return false;
    if (d_mask_u8 && !encode_mask_map(&sm.mask, d_mask_u8, cam->W, cam->H, rgb->n)) return false;
    FwdArgs fa{};
    fa.prm = prm; fa.cam = cam_const(cam);
    fa.rgb = rgb->data; fa.rgb_sn = rgb->sn; fa.dep = depth ? depth->data : nullptr; fa.dep_sn = depth ? depth->sn : 0;
    fa.Hin = cam->H; fa.Win = cam->W; fa.mode_d = depth_mode; fa.mask = d_mask_u8; fa.coverage = d_coverage;
    const dim3 blk(32, 8), grd((cam->W + TILE_W - 1) / TILE_W, (cam->H + TILE_H - 1) / TILE_H, rgb->n);
    if (depth) launch_rgbd_cl<true>(cam, grd, blk, st, fa, sm);
    else launch_rgbd_cl<false>(cam, grd, blk, st, fa, sm);
    return true;                                                   // the caller checks the launch
}

#define VIDC_TRY(expr) do { int rc_ = (expr); if (rc_ != VIDC_OK) return rc_; } while (0)

}  // namespace vidc_k
using namespace vidc_k;

extern "C" __attribute__((visibility("hidden"))) int forward_group(const vidc_camera* cam, const vidc_image* x, const vidc_image* y,
                                                                   vidc_interp mode, vidc_frame_params* d_params_ws, cudaStream_t st);

// ==========================================================================================
extern "C" {

int vidc_abi_version(void) { return VIDC_ABI_VERSION; }
const char* vidc_last_error(void) { return g_err; }
uint64_t vidc_launch_count(void) { return g_launches.load(); }

size_t vidc_workspace_bytes(const vidc_camera* cam, int32_t B) {
    if (!cam || B <= 0 || cam->W <= 0 || cam->H <= 0) return 0;
    const size_t tiles = (size_t)((cam->W + TILE_W - 1) / TILE_W) * (size_t)((cam->H + TILE_H - 1) / TILE_H);
    return (size_t)B * (sizeof(vidc_frame_params) + tiles * sizeof(uint4));
}

int vidc_camera_init(double fx, double fy, double cx, double cy, vidc_camera* cam) {
    if (!cam) return fail(VIDC_ERR_INVALID_ARGUMENT, "null camera");
    if (!(fx != 0.0) || !(fy != 0.0) || !(cx > 0.0) || !(cy > 0.0))
        return fail(VIDC_ERR_INVALID_ARGUMENT, "intrinsics must satisfy fx,fy != 0 and cx,cy > 0");
    cam->W = (int32_t)ceil(2.0 * cx);                                   // :13
    cam->H = (int32_t)ceil(2.0 * cy);                                   // :14
    const double K[9] = {fx, 0, cx, 0, fy, cy, 0, 0, 1};                // :15
    // :16 np.linalg.inv(K) (LAPACK getrf/getri): no pivoting for this upper-triangular K, and
    // trtri forms the last column as -(c * (1/f)).
    const double ifx = 1.0 / fx, ify = 1.0 / fy;
    const double Ki[9] = {ifx, 0, -(cx * ifx), 0, ify, -(cy * ify), 0, 0, 1};
    for (int i = 0; i < 9; ++i) { cam->K[i] = (float)K[i]; cam->Kinv[i] = (float)Ki[i]; }   // :19-20
    cam->cx = (float)cx; cam->cy = (float)cy;
    cam->inv_half_w = (float)(1.0 / ((double)cam->W / 2.0));            // :149
    cam->inv_half_h = (float)(1.0 / ((double)cam->H / 2.0));            // :150
    cam->fx = (float)fx; cam->fy = (float)fy;
    return VIDC_OK;
}

int vidc_frame_params_compute(const vidc_camera* cam, const float* d_Ig, const float* d_Ia, int32_t B,
                              vidc_frame_params* d_params, void* stream) {
    VIDC_TRY(check_cam(cam));
    if (B < 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "negative batch");
    return launch_params(cam, d_Ig, d_Ia, B, d_params, (cudaStream_t)stream);
}

int vidc_frame_params_prepare(const vidc_camera* cam, const float* d_Ig, const float* d_Ia, int32_t B,
                              vidc_frame_params* d_params_ws, float* d_H_out, void* stream) {
    VIDC_TRY(check_cam(cam));
    if (B < 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "negative batch");
    if (tile_skip_enabled() && shear_level() >= 1) return launch_params_tiles(cam, d_Ig, d_Ia, B, d_params_ws, (cudaStream_t)stream, d_H_out);
    return launch_params(cam, d_Ig, d_Ia, B, d_params_ws, (cudaStream_t)stream, d_H_out);
}

int vidc_build_homography(const vidc_camera* cam, const float* d_Ig, const float* d_Ia, int32_t B,
                          float* d_H, float* d_R, float* d_Hinv, void* stream) {
    VIDC_TRY(check_cam(cam));
    if (B < 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "negative batch");
    if (B == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    vidc_frame_params* ws = nullptr;
    VIDC_CUDA(cudaMallocAsync(&ws, sizeof(vidc_frame_params) * (size_t)B, st));
    int rc = launch_params(cam, d_Ig, d_Ia, B, ws, st);
    if (rc == VIDC_OK) rc = scatter_h(ws, B, d_H, d_R, d_Hinv, nullptr, st);
    cudaFreeAsync(ws, st);
    return rc;
}

int vidc_warp_forward(const vidc_camera* cam, const vidc_image* x, const float* d_Ig, const float* d_Ia,
                      int32_t B_gravity, vidc_interp mode, vidc_frame_params* d_params_ws,
                      float* d_H_out, const vidc_image* y, void* stream) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(x, "x", 1, 1 << 30));
    VIDC_TRY(check_image(y, "y", 1, 1 << 30));
    if (x->n != B_gravity) return fail(VIDC_ERR_BATCH_MISMATCH, "x.shape[0]=%d != I_g.shape[0]=%d", x->n, B_gravity);
    if (mode != VIDC_BILINEAR && mode != VIDC_NEAREST && mode != VIDC_BICUBIC) return fail(VIDC_ERR_INVALID_ARGUMENT, "unknown interp mode %d", (int)mode);
    VIDC_TRY(check_out(cam, x, y, "y"));
    if (x->n == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (tile_skip_enabled() && shear_level() >= 1) VIDC_TRY(launch_params_tiles(cam, d_Ig, d_Ia, x->n, d_params_ws, st, d_H_out));
    else VIDC_TRY(launch_params(cam, d_Ig, d_Ia, x->n, d_params_ws, st, d_H_out));
    // F.grid_sample takes any channel count (feature maps): more than four channels go through the kernels in groups of <= 4
    // planes that share the frame parameters computed above
    if (x->c > 4) {
        for (int c0 = 0; c0 < x->c; c0 += 4) {
            vidc_image xg = *x, yg = *y;
            xg.data = x->data + (int64_t)c0 * x->sc; yg.data = y->data + (int64_t)c0 * y->sc;
            xg.c = yg.c = std::min(4, x->c - c0);
            VIDC_TRY(forward_group(cam, &xg, &yg, mode, d_params_ws, st));
        }
        return VIDC_OK;
    }
    return forward_group(cam, x, y, mode, d_params_ws, st);
}

// one group of 1..4 planes of vidc_warp_forward; the frame parameters are already in d_params_ws (not exported)
__attribute__((visibility("hidden"))) int forward_group(const vidc_camera* cam, const vidc_image* x, const vidc_image* y, vidc_interp mode,
                  vidc_frame_params* d_params_ws, cudaStream_t st) {
    if (x->c == 3 && mode == VIDC_BILINEAR && try_rgbd_cl(cam, d_params_ws, x, nullptr, 0, y, nullptr, nullptr, nullptr, st)) {
        VIDC_LAUNCH_CHECK();                                       // channels-last RGB (kernels_shear_cl.cuh)
        return VIDC_OK;
    }
    // contiguous planes of a compile-time geometry: sheared segments (kernels_shear.cuh)
    if (shear_level() >= 1 && mode != VIDC_BICUBIC && (x->c == 1 || x->c == 3) && x->sw == 1 && y->sw == 1 && aligned16(y->data) && y->sn % 4 == 0) {
        auto planes = [&](int Wg, int Hg) {
            const int64_t hw = (int64_t)Wg * Hg;
            return cam->W == Wg && cam->H == Hg && x->w == Wg && x->h == Hg && x->sh == Wg && y->sh == Wg &&
                   (x->c == 1 || (x->sc == hw && y->sc == hw));
        };
        const dim3 blk(32, 8), grd((cam->W + TILE_W - 1) / TILE_W, (cam->H + TILE_H - 1) / TILE_H, x->n);
        PlanesArgs pa;
        pa.prm = d_params_ws; pa.cam = cam_const(cam);
        pa.x = x->data; pa.x_sn = x->sn; pa.y = y->data; pa.y_sn = y->sn; pa.mode = (int)mode;
        pa.src_boxes = nullptr; pa.pf_x = pa.pf_y = pa.pf_z = 0;
        if (tile_skip_enabled() && fwd_prefetch_pct() > 0 && (size_t)grd.x * grd.y <= 320) {     // the tiles kernel wrote the boxes
            static const int sms = [] { int dev = 0, n = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); return n; }();
            const int wave = (int)((long long)sms * VIDC_SHEAR_BLOCKS_FWD * fwd_prefetch_pct() / 100);
            pa.src_boxes = reinterpret_cast<const uint4*>(d_params_ws + x->n);
            pa.pf_x = wave % (int)grd.x; pa.pf_y = (wave / (int)grd.x) % (int)grd.y; pa.pf_z = wave / (int)(grd.x * grd.y);
        }
        bool done = true;
        const bool geom = planes(640, 480) || planes(320, 240) || planes(640, 489) || (cam->W % 32 == 0 && planes(cam->W, cam->H));
        StoreMaps sm;
        const bool ts = geom && tma_store_enabled() &&
                        encode_store_map(&sm.img, y->data, cam->W, cam->H, x->c, x->n, y->sh, x->c == 1 ? (int64_t)cam->W * cam->H : y->sc, y->sn);
        if (planes(640, 480)) launch_planes_shear<640, 480>(x->c, ts, grd, blk, st, pa, sm);
        else if (planes(320, 240)) launch_planes_shear<320, 240>(x->c, ts, grd, blk, st, pa, sm);
        else if (planes(640, 489)) launch_planes_shear<640, 489>(x->c, ts, grd, blk, st, pa, sm);      // the real Azure Kinect canvas: ceil(2 cy) = 489
        else if (geom) launch_planes_shear<0, 0>(x->c, ts, grd, blk, st, pa, sm);                      // any other canvas, runtime geometry
        else done = false;
        if (done) {
            VIDC_LAUNCH_CHECK();
            return VIDC_OK;
        }
    }
    switch (x->c) {
        case 1: return launch_forward<1, false, false>(cam, d_params_ws, x, y, mode, nullptr, nullptr, 0, nullptr, nullptr, st);
        case 2: return launch_forward<2, false, false>(cam, d_params_ws, x, y, mode, nullptr, nullptr, 0, nullptr, nullptr, st);
        case 3: return launch_forward<3, false, false>(cam, d_params_ws, x, y, mode, nullptr, nullptr, 0, nullptr, nullptr, st);
        default: return launch_forward<4, false, false>(cam, d_params_ws, x, y, mode, nullptr, nullptr, 0, nullptr, nullptr, st);
    }
}

// zero_depth_out (sparse-depth path, depth == NULL): a (B,1,H,W) plane the call fills with zeros -- by the RGB kernel's own
// write-out where the sheared kernels run, by a memset otherwise
__attribute__((visibility("hidden"))) int warp_rgbd_impl(const vidc_camera* cam, const vidc_image* rgb, const vidc_image* depth,
                   const float* d_Ig, const float* d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                   vidc_frame_params* d_params_ws, float* d_H_out,
                   const vidc_image* rgb_out, const vidc_image* depth_out,
                   uint8_t* d_mask_u8, uint32_t* d_coverage, const vidc_image* zero_depth_out, void* stream);

int vidc_warp_rgbd(const vidc_camera* cam, const vidc_image* rgb, const vidc_image* depth,
                   const float* d_Ig, const float* d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                   vidc_frame_params* d_params_ws, float* d_H_out,
                   const vidc_image* rgb_out, const vidc_image* depth_out,
                   uint8_t* d_mask_u8, uint32_t* d_coverage, void* stream) {
    return warp_rgbd_impl(cam, rgb, depth, d_Ig, d_Ia, B_gravity, depth_mode, d_params_ws, d_H_out, rgb_out, depth_out, d_mask_u8,
                          d_coverage, nullptr, stream);
}

int warp_rgbd_impl(const vidc_camera* cam, const vidc_image* rgb, const vidc_image* depth,
                   const float* d_Ig, const float* d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                   vidc_frame_params* d_params_ws, float* d_H_out,
                   const vidc_image* rgb_out, const vidc_image* depth_out,
                   uint8_t* d_mask_u8, uint32_t* d_coverage, const vidc_image* zero_depth_out, void* stream) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(rgb, "rgb", 3, 3));
    VIDC_TRY(check_image(rgb_out, "rgb_out", 3, 3));
    if (rgb->n != B_gravity) return fail(VIDC_ERR_BATCH_MISMATCH, "rgb.shape[0]=%d != I_g.shape[0]=%d", rgb->n, B_gravity);
    VIDC_TRY(check_out(cam, rgb, rgb_out, "rgb_out"));
    if (depth) {
        VIDC_TRY(check_image(depth, "depth", 1, 1));
        if (!depth_out) return fail(VIDC_ERR_INVALID_ARGUMENT, "depth given without depth_out");
        VIDC_TRY(check_image(depth_out, "depth_out", 1, 1));
        if (depth->n != rgb->n) return fail(VIDC_ERR_BATCH_MISMATCH, "depth.shape[0]=%d != rgb.shape[0]=%d", depth->n, rgb->n);
        VIDC_TRY(check_out(cam, depth, depth_out, "depth_out"));
        if (depth_mode != VIDC_BILINEAR && depth_mode != VIDC_NEAREST)
            return fail(VIDC_ERR_INVALID_ARGUMENT, "unknown interp mode %d", (int)depth_mode);
    }
    if (rgb->n == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (d_coverage) VIDC_CUDA(cudaMemsetAsync(d_coverage, 0, sizeof(uint32_t) * (size_t)rgb->n, st));
    if (!d_Ig && !d_Ia) VIDC_TRY(prepared_params(d_params_ws, rgb->n, d_H_out, st));
    else if (tile_skip_enabled() && shear_level() >= 1) VIDC_TRY(launch_params_tiles(cam, d_Ig, d_Ia, rgb->n, d_params_ws, st, d_H_out));
    else VIDC_TRY(launch_params(cam, d_Ig, d_Ia, rgb->n, d_params_ws, st, d_H_out));
    if (!zero_depth_out && try_rgbd_cl(cam, d_params_ws, rgb, depth, (int)depth_mode, rgb_out, depth_out, d_mask_u8, d_coverage, st)) {
        VIDC_LAUNCH_CHECK();                                       // channels-last RGB (kernels_shear_cl.cuh)
        return VIDC_OK;
    }
    const bool fast = rgb->sw == 1 && rgb_out->sw == 1 &&
                      (!depth || (depth->sw == 1 && depth_out->sw == 1 && depth->h == rgb->h && depth->w == rgb->w &&
                                  depth->sh == rgb->sh));
    if (fast) {
        const dim3 blk(32, 8), grd((cam->W + TILE_W - 1) / TILE_W, (cam->H + TILE_H - 1) / TILE_H, rgb->n);
        FwdArgs fa;
        fa.prm = d_params_ws; fa.cam = cam_const(cam);
        fa.rgb = rgb->data; fa.rgb_sn = rgb->sn; fa.rgb_sc = (int)rgb->sc;
        fa.dep = depth ? depth->data : nullptr; fa.dep_sn = depth ? depth->sn : 0;
        fa.Hin = rgb->h; fa.Win = rgb->w; fa.in_sh = (int)rgb->sh;
        fa.rgb_o = rgb_out->data; fa.rgbo_sn = rgb_out->sn; fa.rgbo_sc = (int)rgb_out->sc; fa.rgbo_sh = (int)rgb_out->sh;
        fa.dep_o = depth ? depth_out->data : nullptr; fa.depo_sn = depth ? depth_out->sn : 0; fa.depo_sh = depth ? (int)depth_out->sh : 0;
        fa.mode_d = (int)depth_mode; fa.mask = d_mask_u8; fa.coverage = d_coverage;
        fa.src_boxes = nullptr; fa.pf_x = fa.pf_y = fa.pf_z = 0;
        if (tile_skip_enabled() && shear_level() >= 1 && fwd_prefetch_pct() > 0 && (size_t)grd.x * grd.y <= 320) {
            static const int sms = [] { int dev = 0, n = 148; cudaGetDevice(&dev); cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev); return n; }();
            const int wave = (int)((long long)sms * VIDC_SHEAR_BLOCKS_FWD * fwd_prefetch_pct() / 100);
            fa.src_boxes = reinterpret_cast<const uint4*>(d_params_ws + rgb->n);
            fa.pf_x = wave % (int)grd.x; fa.pf_y = (wave / (int)grd.x) % (int)grd.y; fa.pf_z = wave / (int)(grd.x * grd.y);
        }
        // compile-time geometry when input and canvas are contiguous W x H planes of a known size
        auto planes = [&](int Wg, int Hg) {
            return cam->W == Wg && cam->H == Hg && rgb->w == Wg && rgb->h == Hg && rgb->sh == Wg && rgb->sc == (int64_t)Wg * Hg &&
                   rgb_out->sh == Wg && rgb_out->sc == (int64_t)Wg * Hg && (!depth || (depth->sh == Wg && depth_out->sh == Wg));
        };
        if (tma_enabled() && rgb->n > 0) {   // TMA-staged variant: footprint boxes through shared memory
            TmaMaps maps;
            bool ok = true;
            for (int c = 0; c < TMA_NH && ok; ++c) {
                ok = encode_image_map(&maps.a[c], rgb, tma_box_h(c));
                if (ok && depth) ok = encode_image_map(&maps.d[c], depth, tma_box_h(c));
            }
            if (ok) {
                const size_t smem = (size_t)TMA_BW * TMA_BH_MAX * 4 * (depth ? 4 : 3);
                const dim3 tgrd((cam->W + 31) / 32, (cam->H + TMA_TILE_H - 1) / TMA_TILE_H, rgb->n);
                // function attributes belong to the device's context: set on every launch of this opt-in path (cheap)
                if (depth) {
                    cudaFuncSetAttribute(warp_rgbd_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_BW * TMA_BH_MAX * 16);
                    warp_rgbd_tma_kernel<true><<<tgrd, blk, smem, st>>>(fa, maps);
                } else {
                    cudaFuncSetAttribute(warp_rgbd_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TMA_BW * TMA_BH_MAX * 12);
                    warp_rgbd_tma_kernel<false><<<tgrd, blk, smem, st>>>(fa, maps);
                }
                VIDC_LAUNCH_CHECK();
                return VIDC_OK;
            }
        }
        const bool zero_ok = !zero_depth_out || (zero_depth_out->sw == 1 && zero_depth_out->sh == cam->W && aligned16(zero_depth_out->data) &&
                                                  zero_depth_out->sn % 4 == 0);
        const bool shear = shear_level() >= 1 && aligned16(rgb_out->data) && rgb_out->sn % 4 == 0 && zero_ok &&
                           (!depth || (aligned16(depth_out->data) && depth_out->sn % 4 == 0)) &&
                           (!d_mask_u8 || (reinterpret_cast<uintptr_t>(d_mask_u8) & 3) == 0);
        const bool shear_geom = shear && (planes(640, 480) || planes(320, 240) || planes(640, 489) || (cam->W % 32 == 0 && planes(cam->W, cam->H)));
        if (zero_depth_out) {
            if (shear_geom && !tma_enabled()) { fa.dep_o = zero_depth_out->data; fa.depo_sn = zero_depth_out->sn; }     // fused into the write-out
            else {
                if (zero_depth_out->sw != 1 || zero_depth_out->sh != cam->W || zero_depth_out->sn != (int64_t)cam->W * cam->H)
                    return fail(VIDC_ERR_INVALID_ARGUMENT, "depth_out: the sparse-depth path needs a contiguous (B,1,H,W) output");
                VIDC_CUDA(cudaMemsetAsync(zero_depth_out->data, 0, sizeof(float) * (size_t)rgb->n * cam->W * cam->H, st));
            }
        }
        StoreMaps sm;
        bool ts = shear_geom && tma_store_enabled() &&
                  encode_store_map(&sm.img, rgb_out->data, cam->W, cam->H, 3, rgb->n, rgb_out->sh, rgb_out->sc, rgb_out->sn);
        if (ts && depth) ts = encode_store_map(&sm.dep, depth_out->data, cam->W, cam->H, 1, rgb->n, depth_out->sh, (int64_t)cam->W * cam->H, depth_out->sn, true);
        if (ts && zero_depth_out)                                 // sparse-depth route: the zero plane leaves through the same store
            ts = encode_store_map(&sm.dep, zero_depth_out->data, cam->W, cam->H, 1, rgb->n, zero_depth_out->sh, (int64_t)cam->W * cam->H, zero_depth_out->sn, true);
        if (ts && d_mask_u8) ts = encode_mask_map(&sm.mask, d_mask_u8, cam->W, cam->H, rgb->n);
        if (shear && planes(640, 480)) {
            launch_rgbd_shear<640, 480>(depth != nullptr, ts, grd, blk, st, fa, sm);
        } else if (shear && planes(320, 240)) {
            launch_rgbd_shear<320, 240>(depth != nullptr, ts, grd, blk, st, fa, sm);
        } else if (shear && planes(640, 489)) {                            // the real Azure Kinect canvas: ceil(2 cy) = 489
            launch_rgbd_shear<640, 489>(depth != nullptr, ts, grd, blk, st, fa, sm);
        } else if (shear && cam->W % 32 == 0 && planes(cam->W, cam->H)) {  // any other canvas, runtime geometry
            launch_rgbd_shear<0, 0>(depth != nullptr, ts, grd, blk, st, fa, sm);
        } else if (planes(640, 480)) {
            if (depth) warp_rgbd_fast_kernel<640, 480, true><<<grd, blk, 0, st>>>(fa);
            else warp_rgbd_fast_kernel<640, 480, false><<<grd, blk, 0, st>>>(fa);
        } else if (planes(320, 240)) {
            if (depth) warp_rgbd_fast_kernel<320, 240, true><<<grd, blk, 0, st>>>(fa);
            else warp_rgbd_fast_kernel<320, 240, false><<<grd, blk, 0, st>>>(fa);
        } else {
            if (depth) warp_rgbd_fast_kernel<0, 0, true><<<grd, blk, 0, st>>>(fa);
            else warp_rgbd_fast_kernel<0, 0, false><<<grd, blk, 0, st>>>(fa);
        }
        VIDC_LAUNCH_CHECK();
        return VIDC_OK;
    }
    if (zero_depth_out) {
        if (zero_depth_out->sw != 1 || zero_depth_out->sh != cam->W || zero_depth_out->sn != (int64_t)cam->W * cam->H)
            return fail(VIDC_ERR_INVALID_ARGUMENT, "depth_out: the sparse-depth path needs a contiguous (B,1,H,W) output");
        VIDC_CUDA(cudaMemsetAsync(zero_depth_out->data, 0, sizeof(float) * (size_t)rgb->n * cam->W * cam->H, st));
    }
    if (depth)
        return launch_forward<3, true, false>(cam, d_params_ws, rgb, rgb_out, VIDC_BILINEAR, depth, depth_out, depth_mode,
                                              d_mask_u8, d_coverage, st);
    return launch_forward<3, false, false>(cam, d_params_ws, rgb, rgb_out, VIDC_BILINEAR, nullptr, nullptr, 0, d_mask_u8,
                                           d_coverage, st);
}

int vidc_warp_normals_forward(const vidc_camera* cam, const vidc_image* x, const float* d_Ig, const float* d_Ia,
                              int32_t B_gravity, vidc_interp mode, vidc_frame_params* d_params_ws,
                              float* d_H_out, const vidc_image* z, void* stream) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(x, "x", 3, 3));
    VIDC_TRY(check_image(z, "z", 3, 3));
    if (x->n != B_gravity) return fail(VIDC_ERR_BATCH_MISMATCH, "x.shape[0]=%d != I_g.shape[0]=%d", x->n, B_gravity);
    if (mode != VIDC_BILINEAR && mode != VIDC_NEAREST && mode != VIDC_BICUBIC) return fail(VIDC_ERR_INVALID_ARGUMENT, "unknown interp mode %d", (int)mode);
    VIDC_TRY(check_out(cam, x, z, "z"));
    if (x->n == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    VIDC_TRY(launch_params(cam, d_Ig, d_Ia, x->n, d_params_ws, st, d_H_out));
    return launch_forward<3, false, true>(cam, d_params_ws, x, z, mode, nullptr, nullptr, 0, nullptr, nullptr, st);
}

int vidc_warp_with_homography(const vidc_camera* cam, const vidc_image* x, const float* d_Hm, int32_t B_h,
                              vidc_frame_params* d_params_ws, const vidc_image* y, void* stream) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(x, "x", 1, 4));
    VIDC_TRY(check_image(y, "y", 1, 4));
    if (x->n != B_h) return fail(VIDC_ERR_BATCH_MISMATCH, "x.shape[0]=%d != H.shape[0]=%d", x->n, B_h);
    VIDC_TRY(check_out(cam, x, y, "y"));
    if (x->n == 0) return VIDC_OK;
    if (!d_Hm || !d_params_ws) return fail(VIDC_ERR_INVALID_ARGUMENT, "null homography / params pointer");
    cudaStream_t st = (cudaStream_t)stream;
    frame_params_from_h_kernel<<<(x->n + 63) / 64, 64, 0, st>>>(*cam, d_Hm, x->n, d_params_ws);
    VIDC_LAUNCH_CHECK();
    switch (x->c) {
        case 1: return launch_forward<1, false, false>(cam, d_params_ws, x, y, VIDC_BILINEAR, nullptr, nullptr, 0, nullptr, nullptr, st);
        case 2: return launch_forward<2, false, false>(cam, d_params_ws, x, y, VIDC_BILINEAR, nullptr, nullptr, 0, nullptr, nullptr, st);
        case 3: return launch_forward<3, false, false>(cam, d_params_ws, x, y, VIDC_BILINEAR, nullptr, nullptr, 0, nullptr, nullptr, st);
        default: return launch_forward<4, false, false>(cam, d_params_ws, x, y, VIDC_BILINEAR, nullptr, nullptr, 0, nullptr, nullptr, st);
    }
}

int vidc_unwarp_normals(const vidc_camera* cam, const vidc_image* x, const float* d_Ig, const float* d_Ia,
                        int32_t B_gravity, int32_t normalize, vidc_frame_params* d_params_ws,
                        float* d_H_out, const vidc_image* z, uint8_t* d_valid_u8, void* stream) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(x, "x", 3, 3));
    VIDC_TRY(check_image(z, "z", 3, 3));
    if (x->n != B_gravity) return fail(VIDC_ERR_BATCH_MISMATCH, "x.shape[0]=%d != I_g.shape[0]=%d", x->n, B_gravity);
    if (x->h != cam->H || x->w != cam->W)   // reference: .view at :252-254 requires the canvas size
        return fail(VIDC_ERR_INVALID_ARGUMENT, "x must be (B,3,%d,%d), got (%d,%d,%d,%d)", cam->H, cam->W, x->n, x->c, x->h, x->w);
    VIDC_TRY(check_out(cam, x, z, "z"));
    if (x->n == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 blk(32, 8), grd((cam->W + TILE_W - 1) / TILE_W, (cam->H + TILE_H - 1) / TILE_H, x->n);
    InvArgs ia;
    ia.prm = d_params_ws; ia.cam = cam_const(cam);
    ia.x = x->data; ia.x_sn = x->sn; ia.x_sc = (int)x->sc; ia.x_sh = (int)x->sh;
    ia.z = z->data; ia.z_sn = z->sn; ia.z_sc = (int)z->sc; ia.z_sh = (int)z->sh;
    ia.valid = d_valid_u8;
    auto planes = [&](int Wg, int Hg) {
        return cam->W == Wg && cam->H == Hg && x->sh == Wg && x->sc == (int64_t)Wg * Hg && z->sh == Wg && z->sc == (int64_t)Wg * Hg;
    };
    // footprint staged in shared memory (kernels_box.cuh): contiguous planes, rows that are whole float4s
    if (inv_box_enabled() && !tma_enabled() && d_Ig && d_Ia && x->sw == 1 && z->sw == 1 && cam->W % 4 == 0 && planes(cam->W, cam->H) &&
        aligned16(x->data) && x->sn % 4 == 0 && grd.x * grd.y <= 65535u) {     // (not with a prepared workspace: the table would go into it)
        // the per-tile box table lives behind the B parameter blocks of the caller's workspace (vidc_workspace_bytes)
        uint4* boxes = reinterpret_cast<uint4*>(d_params_ws + x->n);
        frame_params_inv_boxes_kernel<<<x->n, 320, 0, st>>>(*cam, d_Ig, d_Ia, x->n, d_params_ws, d_H_out, boxes, (int)grd.x, (int)grd.y);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (planes(640, 480)) launch_unwarp_box<640, 480>(normalize != 0, d_valid_u8 != nullptr, grd, blk, st, ia, boxes);
        else if (planes(320, 240)) launch_unwarp_box<320, 240>(normalize != 0, d_valid_u8 != nullptr, grd, blk, st, ia, boxes);
        else launch_unwarp_box<0, 0>(normalize != 0, d_valid_u8 != nullptr, grd, blk, st, ia, boxes);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        const cudaError_t le = cudaGetLastError();
        if (le != cudaSuccess) return fail(VIDC_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(le));
        return VIDC_OK;
    }
    if (!d_Ig && !d_Ia) VIDC_TRY(prepared_params(d_params_ws, x->n, d_H_out, st));
    else VIDC_TRY(launch_params(cam, d_Ig, d_Ia, x->n, d_params_ws, st, d_H_out));
    if (shear_level() >= 2 && tma_store_enabled() && !d_valid_u8 && cam->W % 32 == 0 && is_channels_last3(x, cam->W, cam->H) &&
        is_channels_last3(z, cam->W, cam->H)) {                    // channels-last normals (kernels_shear_cl.cuh)
        ClStoreMaps sm;
        if (encode_cl_map(&sm.img, z->data, cam->W, cam->H, x->n)) {
            if (normalize) launch_unwarp_cl<true>(cam, grd, blk, st, ia, sm);
            else launch_unwarp_cl<false>(cam, grd, blk, st, ia, sm);
            VIDC_LAUNCH_CHECK();
            return VIDC_OK;
        }
    }
    if (x->sw == 1 && z->sw == 1) {
        if (tma_enabled() && x->n > 0) {
            InvTmaMaps maps;
            bool ok = true;
            for (int c = 0; c < INV_NH && ok; ++c) ok = encode_image_map(&maps.m[c], x, inv_box_h(c), INV_BW);
            if (ok) {
                const int tiles_x = (cam->W + 31) / 32, tiles_y = (cam->H + 31) / 32;
                const long long n_tiles = (long long)tiles_x * tiles_y * x->n;
                int dev = 0, sms = 148;
                cudaGetDevice(&dev);
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
                const int ctas = (int)std::min<long long>(n_tiles, (long long)sms * 4);
                const size_t smem = sizeof(float) * INV_STAGE_FLOATS * INV_STAGES;
                if (normalize) {
                    cudaFuncSetAttribute(unwarp_normals_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(float) * INV_STAGE_FLOATS * INV_STAGES));
                    unwarp_normals_tma_kernel<true><<<ctas, 288, smem, st>>>(ia, maps, tiles_x, tiles_y, (int)n_tiles);
                } else {
                    cudaFuncSetAttribute(unwarp_normals_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(float) * INV_STAGE_FLOATS * INV_STAGES));
                    unwarp_normals_tma_kernel<false><<<ctas, 288, smem, st>>>(ia, maps, tiles_x, tiles_y, (int)n_tiles);
                }
                VIDC_LAUNCH_CHECK();
                return VIDC_OK;
            }
        }
        const bool shear = shear_level() >= 2 && aligned16(z->data) && z->sn % 4 == 0 &&
                           (!d_valid_u8 || (reinterpret_cast<uintptr_t>(d_valid_u8) & 3) == 0);
        StoreMaps sm;
        const bool ts = shear && tma_store_enabled() && !d_valid_u8 && cam->W % 32 == 0 && planes(cam->W, cam->H) &&
                        encode_store_map(&sm.img, z->data, cam->W, cam->H, 3, x->n, z->sh, z->sc, z->sn);
        if (shear && planes(640, 480)) {
            launch_unwarp_shear<640, 480>(normalize != 0, d_valid_u8 != nullptr, ts, grd, blk, st, ia, sm);
        } else if (shear && planes(320, 240)) {
            launch_unwarp_shear<320, 240>(normalize != 0, d_valid_u8 != nullptr, ts, grd, blk, st, ia, sm);
        } else if (shear && planes(640, 489)) {
            launch_unwarp_shear<640, 489>(normalize != 0, d_valid_u8 != nullptr, ts, grd, blk, st, ia, sm);
        } else if (shear && cam->W % 32 == 0 && planes(cam->W, cam->H)) {  // any other canvas, runtime geometry
            launch_unwarp_shear<0, 0>(normalize != 0, d_valid_u8 != nullptr, ts, grd, blk, st, ia, sm);
        } else if (planes(640, 480)) {
            if (normalize) unwarp_normals_fast_kernel<640, 480, true><<<grd, blk, 0, st>>>(ia);
            else unwarp_normals_fast_kernel<640, 480, false><<<grd, blk, 0, st>>>(ia);
        } else if (planes(320, 240)) {
            if (normalize) unwarp_normals_fast_kernel<320, 240, true><<<grd, blk, 0, st>>>(ia);
            else unwarp_normals_fast_kernel<320, 240, false><<<grd, blk, 0, st>>>(ia);
        } else {
            if (normalize) unwarp_normals_fast_kernel<0, 0, true><<<grd, blk, 0, st>>>(ia);
            else unwarp_normals_fast_kernel<0, 0, false><<<grd, blk, 0, st>>>(ia);
        }
        VIDC_LAUNCH_CHECK();
        return VIDC_OK;
    }
    if (normalize)
        unwarp_normals_kernel<true><<<grid2d(cam->W, cam->H, x->n, blk), blk, 0, st>>>(d_params_ws, cam_const(cam), view_in(x), view_out(z), d_valid_u8);
    else
        unwarp_normals_kernel<false><<<grid2d(cam->W, cam->H, x->n, blk), blk, 0, st>>>(d_params_ws, cam_const(cam), view_in(x), view_out(z), d_valid_u8);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_sampler_forward_inverse(const vidc_camera* cam, const float* d_Ig, const float* d_Ia, int32_t B,
                                 vidc_frame_params* d_params_ws, float* d_Rt, float* d_grid,
                                 float* d_inv_grid, void* stream) {
    VIDC_TRY(check_cam(cam));
    if (B < 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "negative batch");
    if (B == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    VIDC_TRY(launch_params(cam, d_Ig, d_Ia, B, d_params_ws, st));
    if (d_Rt) {
        guard_rt_kernel<<<(B * 9 + 127) / 128, 128, 0, st>>>(d_params_ws, B, d_Rt);
        VIDC_LAUNCH_CHECK();
    }
    if (d_grid || d_inv_grid) {
        const dim3 blk(32, 8);
        sampler_grids_kernel<<<grid2d(cam->W, cam->H, B, blk), blk, 0, st>>>(d_params_ws, cam_const(cam), (float2*)d_grid, (float2*)d_inv_grid);
        VIDC_LAUNCH_CHECK();
    }
    return VIDC_OK;
}

int vidc_validity_mask(const vidc_image* x1, uint8_t* d_mask_u8, float* d_mask_f32, uint32_t* d_coverage, void* stream) {
    VIDC_TRY(check_image(x1, "x1", 3, 1 << 30));
    if (x1->n == 0) return VIDC_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (d_coverage) VIDC_CUDA(cudaMemsetAsync(d_coverage, 0, sizeof(uint32_t) * (size_t)x1->n, st));
    const long long hw = (long long)x1->h * x1->w;
    if (x1->sw == 1 && x1->sh == x1->w && x1->sc == hw && hw % 4 == 0 && x1->sn % 4 == 0 && aligned16(x1->data) &&
        (!d_mask_f32 || aligned16(d_mask_f32)) && (!d_mask_u8 || (reinterpret_cast<uintptr_t>(d_mask_u8) & 3) == 0)) {
        const int hw4 = (int)(hw / 4);
        const dim3 grd((unsigned)std::min<long long>((hw4 + 255) / 256, 1184), x1->n);        // 8 CTAs x 148 SMs per frame at most
        validity_mask_vec4_kernel<<<grd, 256, 0, st>>>(x1->data, x1->sn, hw4, d_mask_u8, d_mask_f32, d_coverage);
        VIDC_LAUNCH_CHECK();
        return VIDC_OK;
    }
    const dim3 blk(32, 8);
    validity_mask_kernel<<<grid2d(x1->w, x1->h, x1->n, blk), blk, 0, st>>>(view_in(x1), d_mask_u8, d_mask_f32, d_coverage);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_mask_nearest(const float* d_mask, int32_t B, int32_t Hin, int32_t Win, int32_t Hout, int32_t Wout,
                      float* d_out, void* stream) {
    if (B < 0 || Hin <= 0 || Win <= 0 || Hout <= 0 || Wout <= 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "bad mask sizes");
    if (B == 0) return VIDC_OK;
    if (!d_mask || !d_out) return fail(VIDC_ERR_INVALID_ARGUMENT, "null mask pointer");
    const long long total = (long long)B * Hout * Wout;
    mask_nearest_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_mask, B, Hin, Win, Hout, Wout, d_out);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_mask_pyramid(const uint8_t* d_mask_u8, const float* d_mask_f32, int32_t B, int32_t Hin, int32_t Win,
                      int32_t levels, const int32_t* sizes_hw, float* const* d_outs, void* stream) {
    if (B < 0 || Hin <= 0 || Win <= 0 || levels < 1 || levels > 4 || !sizes_hw || !d_outs)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "bad pyramid request (1..4 levels)");
    if (!d_mask_u8 == !d_mask_f32) return fail(VIDC_ERR_INVALID_ARGUMENT, "exactly one of the u8 / f32 source masks must be given");
    if (B == 0) return VIDC_OK;
    PyramidArgs pa;
    pa.m8 = d_mask_u8; pa.m32 = d_mask_f32; pa.B = B; pa.Hin = Hin; pa.Win = Win; pa.levels = levels;
    pa.begin[0] = 0;
    for (int l = 0; l < 4; ++l) {
        const bool on = l < levels;
        pa.Ho[l] = on ? sizes_hw[2 * l] : 1; pa.Wo[l] = on ? sizes_hw[2 * l + 1] : 1; pa.out[l] = on ? d_outs[l] : nullptr;
        if (on && (pa.Ho[l] <= 0 || pa.Wo[l] <= 0 || !pa.out[l])) return fail(VIDC_ERR_INVALID_ARGUMENT, "bad pyramid level %d", l);
        pa.begin[l + 1] = pa.begin[l] + (on ? (long long)B * pa.Ho[l] * pa.Wo[l] : 0);
    }
    const long long total = pa.begin[levels];
    mask_pyramid_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(pa);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_normalize3(const vidc_image* z, const vidc_image* out, void* stream) {
    VIDC_TRY(check_image(z, "z", 3, 3));
    VIDC_TRY(check_image(out, "out", 3, 3));
    if (out->n != z->n || out->h != z->h || out->w != z->w) return fail(VIDC_ERR_INVALID_ARGUMENT, "normalize3: shape mismatch");
    if (z->n == 0) return VIDC_OK;
    const long long hw = (long long)z->h * z->w;
    if (z->sw == 1 && out->sw == 1 && z->sh == z->w && out->sh == z->w && z->sc == hw && out->sc == hw && hw % 4 == 0 &&
        z->sn % 4 == 0 && out->sn % 4 == 0 && aligned16(z->data) && aligned16(out->data)) {
        const int hw4 = (int)(hw / 4);
        const dim3 grd((unsigned)std::min<long long>((hw4 + 255) / 256, 1184), z->n);
        normalize3_vec4_kernel<<<grd, 256, 0, (cudaStream_t)stream>>>(z->data, z->sn, out->data, out->sn, hw4);
        VIDC_LAUNCH_CHECK();
        return VIDC_OK;
    }
    const dim3 blk(32, 8);
    normalize3_kernel<<<grid2d(z->w, z->h, z->n, blk), blk, 0, (cudaStream_t)stream>>>(view_in(z), view_out(out));
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_normal_stats(const vidc_image* gt, const vidc_image* pred, const vidc_image* mask,
                      int32_t normalize_prediction, double* d_out, void* stream) {
    VIDC_TRY(check_image(gt, "norm_gt", 3, 3));
    VIDC_TRY(check_image(pred, "pred_normals", 3, 1 << 30));
    VIDC_TRY(check_image(mask, "mask", 1, 1));
    if (pred->n != gt->n || mask->n != gt->n || pred->h != gt->h || pred->w != gt->w || mask->h != gt->h || mask->w != gt->w)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "normal_stats: shape mismatch");
    if (!d_out) return fail(VIDC_ERR_INVALID_ARGUMENT, "null output");
    cudaStream_t st = (cudaStream_t)stream;
    VIDC_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double) * 4, st));
    if (gt->n == 0) return VIDC_OK;
    const dim3 blk(32, 8);
    normal_stats_kernel<<<grid2d(gt->w, gt->h, gt->n, blk), blk, 0, st>>>(view_in(gt), view_in(pred), view_in(mask), normalize_prediction, d_out);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_normal_loss_backward(const vidc_image* gt, const vidc_image* pred, const vidc_image* mask, int32_t loss_mode,
                              const double* d_stats, const float* d_grad_loss, const vidc_image* grad_pred, void* stream) {
    VIDC_TRY(check_image(gt, "norm_gt", 3, 3));
    VIDC_TRY(check_image(pred, "pred_normals", 3, 1 << 30));
    VIDC_TRY(check_image(mask, "mask", 1, 1));
    VIDC_TRY(check_image(grad_pred, "grad_pred", 3, 1 << 30));
    if (pred->n != gt->n || mask->n != gt->n || pred->h != gt->h || pred->w != gt->w || mask->h != gt->h || mask->w != gt->w ||
        grad_pred->n != pred->n || grad_pred->c != pred->c || grad_pred->h != pred->h || grad_pred->w != pred->w)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "normal_loss_backward: shape mismatch");
    if (loss_mode < 0 || loss_mode > 2) return fail(VIDC_ERR_INVALID_ARGUMENT, "normal_loss_backward: loss_mode must be 0, 1 or 2");
    if (!d_stats || !d_grad_loss) return fail(VIDC_ERR_INVALID_ARGUMENT, "null stats / grad_loss pointer");
    if (gt->n == 0) return VIDC_OK;
    const dim3 blk(32, 8);
    normal_loss_backward_kernel<<<grid2d(gt->w, gt->h, gt->n, blk), blk, 0, (cudaStream_t)stream>>>(
        view_in(gt), view_in(pred), view_in(mask), loss_mode, d_stats, d_grad_loss, view_out(grad_pred));
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_to_tensor_u8(const uint8_t* d_hwc, int32_t B, int32_t H, int32_t W, int32_t C, float* d_chw, void* stream) {
    if (B < 0 || H <= 0 || W <= 0 || C < 1 || C > 4) return fail(VIDC_ERR_INVALID_ARGUMENT, "to_tensor: bad shape (%d,%d,%d,%d)", B, H, W, C);
    if (B == 0) return VIDC_OK;
    if (!d_hwc || !d_chw) return fail(VIDC_ERR_INVALID_ARGUMENT, "to_tensor: null image pointer");
    if (B > 65535) return fail(VIDC_ERR_INVALID_ARGUMENT, "to_tensor: at most 65535 frames per call");
    const long long hw = (long long)H * W;
    cudaStream_t st = (cudaStream_t)stream;
    if (C == 3 && hw % 4 == 0 && ((uintptr_t)d_hwc & 3) == 0 && aligned16(d_chw))
        to_tensor_rgb_u8_kernel<<<dim3((unsigned)((hw / 4 + 255) / 256), B), 256, 0, st>>>(reinterpret_cast<const uint32_t*>(d_hwc), hw, d_chw);
    else
        to_tensor_u8_kernel<<<dim3((unsigned)((hw + 255) / 256), B), 256, 0, st>>>(d_hwc, hw, C, d_chw);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

// ---- host-buffer end-to-end ---------------------------------------------------------------
// The batch is cut into chunks and software-pipelined over three internal streams so that the H2D copy of
// chunk c+1, the kernels of chunk c and the D2H copy of chunk c-1 overlap (PCIe is full duplex, the copy
// engines run beside the SMs).  Ordering against the caller's stream is by events only.
namespace {
int e2e_chunk() {                       // frames per pipeline stage (VIDC_E2E_CHUNK overrides the default)
    static int v = [] { const char* e = getenv("VIDC_E2E_CHUNK"); int c = e ? atoi(e) : 0; return c > 0 ? c : 16; }();
    return v;
}
constexpr int E2E_MAX_CHUNKS = 4096;
struct Workspace {
    int device = -1;
    size_t cap = 0;          // bytes
    char* base = nullptr;
    cudaStream_t s_in = nullptr, s_comp = nullptr, s_out = nullptr;
    cudaEvent_t ev_start = nullptr, ev_done = nullptr;
    std::vector<cudaEvent_t> ev_in, ev_comp;
};
// One workspace (scratch + three streams + events) PER DEVICE, each behind its own mutex: a process that drives several GPUs
// -- from one thread or from several -- neither serialises its devices on one lock nor tears the scratch down whenever the
// current device changes (round 1 had one global workspace).
constexpr int E2E_MAX_DEVICES = 64;
std::mutex g_ws_mutex[E2E_MAX_DEVICES];
Workspace g_ws_dev[E2E_MAX_DEVICES];

void ws_destroy(Workspace& w) {
    if (w.device < 0) return;
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(w.device);
    if (w.base) cudaFree(w.base);
    if (w.s_in) cudaStreamDestroy(w.s_in);
    if (w.s_comp) cudaStreamDestroy(w.s_comp);
    if (w.s_out) cudaStreamDestroy(w.s_out);
    if (w.ev_start) cudaEventDestroy(w.ev_start);
    if (w.ev_done) cudaEventDestroy(w.ev_done);
    for (cudaEvent_t e : w.ev_in) cudaEventDestroy(e);
    for (cudaEvent_t e : w.ev_comp) cudaEventDestroy(e);
    cudaSetDevice(cur);
    w = Workspace();
}
}  // namespace

int vidc_release_workspace(void) {
    for (int d = 0; d < E2E_MAX_DEVICES; ++d) {
        std::lock_guard<std::mutex> lk(g_ws_mutex[d]);
        ws_destroy(g_ws_dev[d]);
    }
    return VIDC_OK;
}

namespace {
// h_rgb (B,3,H,W) float, or h_rgb_u8 (B,H,W,3) uint8 as the DataLoader decodes it (converted on the device: a quarter of the bytes)
int warp_unwarp_host_impl(const vidc_camera* cam, int32_t B,
                          const float* h_rgb, const uint8_t* h_rgb_u8, const float* h_depth, const float* h_normals,
                          const float* h_Ig, const float* h_Ia,
                          float* h_rgb_w, float* h_depth_w, uint8_t* h_mask, float* h_normals_cam,
                          void* stream);
}  // namespace

int vidc_warp_unwarp_host(const vidc_camera* cam, int32_t B,
                          const float* h_rgb, const float* h_depth, const float* h_normals,
                          const float* h_Ig, const float* h_Ia,
                          float* h_rgb_w, float* h_depth_w, uint8_t* h_mask, float* h_normals_cam,
                          void* stream) {
    if (B > 0 && !h_rgb) return fail(VIDC_ERR_INVALID_ARGUMENT, "null host input");
    return warp_unwarp_host_impl(cam, B, h_rgb, nullptr, h_depth, h_normals, h_Ig, h_Ia, h_rgb_w, h_depth_w, h_mask, h_normals_cam, stream);
}

int vidc_warp_unwarp_host_u8(const vidc_camera* cam, int32_t B,
                             const uint8_t* h_rgb_u8, const float* h_depth, const float* h_normals,
                             const float* h_Ig, const float* h_Ia,
                             float* h_rgb_w, float* h_depth_w, uint8_t* h_mask, float* h_normals_cam,
                             void* stream) {
    if (B > 0 && !h_rgb_u8) return fail(VIDC_ERR_INVALID_ARGUMENT, "null host input");
    return warp_unwarp_host_impl(cam, B, nullptr, h_rgb_u8, h_depth, h_normals, h_Ig, h_Ia, h_rgb_w, h_depth_w, h_mask, h_normals_cam, stream);
}

namespace {
int warp_unwarp_host_impl(const vidc_camera* cam, int32_t B,
                          const float* h_rgb, const uint8_t* h_rgb_u8, const float* h_depth, const float* h_normals,
                          const float* h_Ig, const float* h_Ia,
                          float* h_rgb_w, float* h_depth_w, uint8_t* h_mask, float* h_normals_cam,
                          void* stream) {
    VIDC_TRY(check_cam(cam));
    if (B < 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "negative batch");
    if (B == 0) return VIDC_OK;
    if ((!h_rgb && !h_rgb_u8) || !h_normals || !h_Ig || !h_Ia) return fail(VIDC_ERR_INVALID_ARGUMENT, "null host input");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t hw = (size_t)cam->H * cam->W, fb = hw * sizeof(float);
    auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
    // layout: rgb | depth | normals | rgb_w | depth_w | normals_cam | mask | Ig | Ia | params
    const size_t o_rgb = 0, o_dep = o_rgb + al(3 * fb * B), o_nrm = o_dep + al(fb * B), o_rgbw = o_nrm + al(3 * fb * B),
                 o_depw = o_rgbw + al(3 * fb * B), o_nc = o_depw + al(fb * B), o_mask = o_nc + al(3 * fb * B),
                 o_ig = o_mask + al(hw * B), o_ia = o_ig + al(12 * (size_t)B), o_prm = o_ia + al(12 * (size_t)B),
                 o_u8 = o_prm + al(vidc_workspace_bytes(cam, B)), total = o_u8 + (h_rgb_u8 ? al(3 * hw * B) : 0);
    // Chunk schedule: full chunks in the steady state, a ramp of small chunks at both ends.  The first H2D and the last
    // D2H cannot overlap anything (pipeline fill / drain), so their chunks are kept short: measured 5.23 K -> see
    // profiles/r1_history.md.  VIDC_E2E_RAMP=0 turns the ramp off.
    const int E2E_CHUNK = e2e_chunk();
    std::vector<int> sizes;
    {
        static const bool ramp = [] { const char* e = getenv("VIDC_E2E_RAMP"); return !(e && e[0] == '0'); }();
        std::vector<int> head;
        if (ramp) for (int c = std::max(1, E2E_CHUNK / 8); c < E2E_CHUNK; c *= 2) head.push_back(c);     // 2, 4, 8 for 16
        int head_sum = 0;
        for (int c : head) head_sum += c;
        int left = B;
        if (2 * head_sum + E2E_CHUNK <= B) {
            for (int c : head) sizes.push_back(c);
            left -= 2 * head_sum;
        } else {
            head.clear();
        }
        for (; left > 0; left -= E2E_CHUNK) sizes.push_back(std::min(E2E_CHUNK, left));
        for (auto it = head.rbegin(); it != head.rend(); ++it) sizes.push_back(*it);
    }
    const int nchunks = (int)sizes.size();
    if (nchunks > E2E_MAX_CHUNKS) return fail(VIDC_ERR_INVALID_ARGUMENT, "batch too large for one host call");
    int dev = 0;
    VIDC_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= E2E_MAX_DEVICES) return fail(VIDC_ERR_NO_DEVICE, "device ordinal %d out of range", dev);
    std::lock_guard<std::mutex> lk(g_ws_mutex[dev]);
    Workspace& g_ws = g_ws_dev[dev];
    if (g_ws.device != dev) {
        g_ws.device = dev;
        VIDC_CUDA(cudaStreamCreateWithFlags(&g_ws.s_in, cudaStreamNonBlocking));
        VIDC_CUDA(cudaStreamCreateWithFlags(&g_ws.s_comp, cudaStreamNonBlocking));
        VIDC_CUDA(cudaStreamCreateWithFlags(&g_ws.s_out, cudaStreamNonBlocking));
        VIDC_CUDA(cudaEventCreateWithFlags(&g_ws.ev_start, cudaEventDisableTiming));
        VIDC_CUDA(cudaEventCreateWithFlags(&g_ws.ev_done, cudaEventDisableTiming));
    }
    if (g_ws.cap < total) {
        if (g_ws.base) { cudaFree(g_ws.base); g_ws.base = nullptr; g_ws.cap = 0; }
        VIDC_CUDA(cudaMalloc(&g_ws.base, total));
        g_ws.cap = total;
    }
    while ((int)g_ws.ev_in.size() < nchunks) {
        cudaEvent_t a, b;
        VIDC_CUDA(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        VIDC_CUDA(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        g_ws.ev_in.push_back(a); g_ws.ev_comp.push_back(b);
    }
    char* w = g_ws.base;
    cudaStream_t s_in = g_ws.s_in, s_comp = g_ws.s_comp, s_out = g_ws.s_out;
    // From here on copies target the caller's host buffers: on ANY failure the three internal streams are drained before the
    // error is returned, so the caller may free its buffers as soon as it sees the status.
    const int rc_pipeline = [&]() -> int {
    // everything the caller enqueued before this call happens-before the pipeline
    VIDC_CUDA(cudaEventRecord(g_ws.ev_start, st));
    VIDC_CUDA(cudaStreamWaitEvent(s_in, g_ws.ev_start, 0));
    VIDC_CUDA(cudaStreamWaitEvent(s_out, g_ws.ev_start, 0));
    VIDC_CUDA(cudaMemcpyAsync(w + o_ig, h_Ig, 12 * (size_t)B, cudaMemcpyHostToDevice, s_in));
    VIDC_CUDA(cudaMemcpyAsync(w + o_ia, h_Ia, 12 * (size_t)B, cudaMemcpyHostToDevice, s_in));
    size_t f_next = 0;
    for (int c = 0; c < nchunks; ++c) {
        const size_t f0 = f_next;
        const int n = sizes[c];
        f_next += (size_t)n;
        if (h_rgb_u8) VIDC_CUDA(cudaMemcpyAsync(w + o_u8 + 3 * hw * f0, h_rgb_u8 + 3 * hw * f0, 3 * hw * n, cudaMemcpyHostToDevice, s_in));
        else VIDC_CUDA(cudaMemcpyAsync(w + o_rgb + 3 * fb * f0, h_rgb + 3 * hw * f0, 3 * fb * n, cudaMemcpyHostToDevice, s_in));
        if (h_depth) VIDC_CUDA(cudaMemcpyAsync(w + o_dep + fb * f0, h_depth + hw * f0, fb * n, cudaMemcpyHostToDevice, s_in));
        VIDC_CUDA(cudaMemcpyAsync(w + o_nrm + 3 * fb * f0, h_normals + 3 * hw * f0, 3 * fb * n, cudaMemcpyHostToDevice, s_in));
        VIDC_CUDA(cudaEventRecord(g_ws.ev_in[c], s_in));
        VIDC_CUDA(cudaStreamWaitEvent(s_comp, g_ws.ev_in[c], 0));
        auto img = [&](size_t off, int ch) {
            vidc_image im; im.data = (float*)(w + off) + (size_t)ch * hw * f0; im.n = n; im.c = ch; im.h = cam->H; im.w = cam->W;
            im.sn = (int64_t)ch * hw; im.sc = (int64_t)hw; im.sh = cam->W; im.sw = 1; return im;
        };
        const vidc_image rgb = img(o_rgb, 3), dep = img(o_dep, 1), nrm = img(o_nrm, 3), rgbw = img(o_rgbw, 3),
                         depw = img(o_depw, 1), nc = img(o_nc, 3);
        vidc_frame_params* prm = (vidc_frame_params*)(w + o_prm) + f0;
        const float* ig = (const float*)(w + o_ig) + 3 * f0;
        const float* ia = (const float*)(w + o_ia) + 3 * f0;
        if (h_rgb_u8) VIDC_TRY(vidc_to_tensor_u8((const uint8_t*)(w + o_u8) + 3 * hw * f0, n, cam->H, cam->W, 3, rgb.data, s_comp));
        VIDC_TRY(vidc_frame_params_prepare(cam, ig, ia, n, prm, nullptr, s_comp));      // once per chunk, shared by both directions
        VIDC_TRY(vidc_warp_rgbd(cam, &rgb, h_depth ? &dep : nullptr, nullptr, nullptr, n, VIDC_BILINEAR, prm, nullptr, &rgbw,
                                h_depth ? &depw : nullptr, h_mask ? (uint8_t*)(w + o_mask) + hw * f0 : nullptr, nullptr, s_comp));
        VIDC_TRY(vidc_unwarp_normals(cam, &nrm, nullptr, nullptr, n, 1, prm, nullptr, &nc, nullptr, s_comp));
        VIDC_CUDA(cudaEventRecord(g_ws.ev_comp[c], s_comp));
        VIDC_CUDA(cudaStreamWaitEvent(s_out, g_ws.ev_comp[c], 0));
        if (h_rgb_w) VIDC_CUDA(cudaMemcpyAsync(h_rgb_w + 3 * hw * f0, w + o_rgbw + 3 * fb * f0, 3 * fb * n, cudaMemcpyDeviceToHost, s_out));
        if (h_depth_w && h_depth) VIDC_CUDA(cudaMemcpyAsync(h_depth_w + hw * f0, w + o_depw + fb * f0, fb * n, cudaMemcpyDeviceToHost, s_out));
        if (h_mask) VIDC_CUDA(cudaMemcpyAsync(h_mask + hw * f0, w + o_mask + hw * f0, hw * n, cudaMemcpyDeviceToHost, s_out));
        if (h_normals_cam) VIDC_CUDA(cudaMemcpyAsync(h_normals_cam + 3 * hw * f0, w + o_nc + 3 * fb * f0, 3 * fb * n, cudaMemcpyDeviceToHost, s_out));
    }
    // join: the caller's stream continues after the last D2H (s_out also covers s_comp and s_in transitively)
    VIDC_CUDA(cudaEventRecord(g_ws.ev_done, s_out));
    VIDC_CUDA(cudaStreamWaitEvent(st, g_ws.ev_done, 0));
    VIDC_CUDA(cudaStreamSynchronize(st));
    return VIDC_OK;
    }();
    if (rc_pipeline != VIDC_OK) {
        cudaStreamSynchronize(s_in); cudaStreamSynchronize(s_comp); cudaStreamSynchronize(s_out);
    }
    return rc_pipeline;
}
}  // namespace

int vidc_warp_rgbd_packed(const vidc_camera* cam, const float* d_in, int32_t B, int32_t Hin, int32_t Win,
                          const float* d_Ig, const float* d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                          vidc_frame_params* d_params_ws, float* d_H_out, float* d_out, uint8_t* d_mask_u8,
                          uint32_t* d_coverage, void* stream) {
    VIDC_TRY(check_cam(cam));
    if (B < 0 || Hin <= 0 || Win <= 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "bad packed image shape");
    if (B != B_gravity) return fail(VIDC_ERR_BATCH_MISMATCH, "x.shape[0]=%d != I_g.shape[0]=%d", B, B_gravity);
    if (depth_mode != VIDC_BILINEAR && depth_mode != VIDC_NEAREST) return fail(VIDC_ERR_INVALID_ARGUMENT, "unknown interp mode %d", (int)depth_mode);
    if (B == 0) return VIDC_OK;
    if (!d_in || !d_out) return fail(VIDC_ERR_INVALID_ARGUMENT, "null packed image pointer");
    if (((uintptr_t)d_in & 15) || ((uintptr_t)d_out & 15)) return fail(VIDC_ERR_INVALID_ARGUMENT, "packed images must be 16-byte aligned");
    if ((long long)Hin * Win >= (1LL << 29)) return fail(VIDC_ERR_INVALID_ARGUMENT, "frame too large");
    cudaStream_t st = (cudaStream_t)stream;
    if (d_coverage) VIDC_CUDA(cudaMemsetAsync(d_coverage, 0, sizeof(uint32_t) * (size_t)B, st));
    VIDC_TRY(launch_params(cam, d_Ig, d_Ia, B, d_params_ws, st, d_H_out));
    PackedArgs pa;
    pa.prm = d_params_ws; pa.cam = cam_const(cam);
    pa.in = reinterpret_cast<const float4*>(d_in); pa.in_sn = (long long)Hin * Win; pa.Hin = Hin; pa.Win = Win;
    pa.out = reinterpret_cast<float4*>(d_out); pa.out_sn = (long long)cam->H * cam->W;
    pa.mode_d = (int)depth_mode; pa.mask = d_mask_u8; pa.coverage = d_coverage;
    const dim3 blk(32, 8), grd((cam->W + TILE_W - 1) / TILE_W, (cam->H + TILE_H - 1) / TILE_H, B);
    warp_rgbd_nhwc4_kernel<<<grd, blk, 0, st>>>(pa);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

namespace {
// argument checks shared by the scatter and the ordered backward
int check_warp_backward(const vidc_camera* cam, const vidc_image* grad_out, int32_t B_gravity, int32_t inverse, vidc_interp mode,
                        int32_t Hin, int32_t Win) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(grad_out, "grad_out", 1, 1 << 30));
    if (grad_out->c > 4) return fail(VIDC_ERR_INVALID_ARGUMENT, "grad_out: at most 4 channels per call (3 for the inverse warp); split wider feature maps into groups");
    if (grad_out->n != B_gravity) return fail(VIDC_ERR_BATCH_MISMATCH, "grad.shape[0]=%d != I_g.shape[0]=%d", grad_out->n, B_gravity);
    if (grad_out->h != cam->H || grad_out->w != cam->W) return fail(VIDC_ERR_INVALID_ARGUMENT, "grad_out must have the canvas size");
    if (inverse && (grad_out->c != 3 || Hin != cam->H || Win != cam->W)) return fail(VIDC_ERR_INVALID_ARGUMENT, "inverse backward needs (B,3,H,W)");
    if (mode != VIDC_BILINEAR && mode != VIDC_NEAREST) return fail(VIDC_ERR_INVALID_ARGUMENT, "unknown interp mode %d", (int)mode);
    if (Hin <= 0 || Win <= 0 || (long long)Hin * Win * grad_out->c >= (1LL << 31)) return fail(VIDC_ERR_INVALID_ARGUMENT, "bad input size");
    return VIDC_OK;
}
}  // namespace

int vidc_warp_backward(const vidc_camera* cam, const vidc_image* grad_out, const float* d_Ig, const float* d_Ia,
                       int32_t B_gravity, int32_t inverse, vidc_interp mode, vidc_frame_params* d_params_ws,
                       float* d_grad_in, int32_t Hin, int32_t Win, void* stream) {
    VIDC_TRY(check_warp_backward(cam, grad_out, B_gravity, inverse, mode, Hin, Win));
    if (grad_out->n == 0) return VIDC_OK;
    if (!d_grad_in) return fail(VIDC_ERR_INVALID_ARGUMENT, "null grad_in");
    cudaStream_t st = (cudaStream_t)stream;
    const int C = grad_out->c;
    VIDC_CUDA(cudaMemsetAsync(d_grad_in, 0, sizeof(float) * (size_t)grad_out->n * C * Hin * Win, st));
    VIDC_TRY(launch_params(cam, d_Ig, d_Ia, grad_out->n, d_params_ws, st));
    const dim3 blk(32, 8);
    if (inverse)
        warp_backward_kernel<true><<<grid2d(cam->W, cam->H, grad_out->n, blk), blk, 0, st>>>(d_params_ws, cam_const(cam), view_in(grad_out), C,
                                                                                         (int)mode, d_grad_in, (long long)C * Hin * Win, Hin * Win, Hin, Win);
    else
        warp_backward_kernel<false><<<grid2d(cam->W, cam->H, grad_out->n, blk), blk, 0, st>>>(d_params_ws, cam_const(cam), view_in(grad_out), C,
                                                                                          (int)mode, d_grad_in, (long long)C * Hin * Win, Hin * Win, Hin, Win);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_warp_backward_ordered(const vidc_camera* cam, const vidc_image* grad_out, const float* d_Ig, const float* d_Ia,
                               int32_t B_gravity, int32_t inverse, vidc_interp mode, vidc_frame_params* d_params_ws,
                               float* d_grad_in, int32_t Hin, int32_t Win, void* stream) {
    VIDC_TRY(check_warp_backward(cam, grad_out, B_gravity, inverse, mode, Hin, Win));
    if (grad_out->n == 0) return VIDC_OK;
    if (!d_grad_in) return fail(VIDC_ERR_INVALID_ARGUMENT, "null grad_in");
    cudaStream_t st = (cudaStream_t)stream;
    const int C = grad_out->c;
    VIDC_TRY(launch_params(cam, d_Ig, d_Ia, grad_out->n, d_params_ws, st));
    const dim3 grd((Win + BWO_TILE - 1) / BWO_TILE, (Hin + BWO_TILE - 1) / BWO_TILE, grad_out->n);    // every grad_in element once
    if (inverse)
        warp_backward_ordered_kernel<true><<<grd, 256, 0, st>>>(d_params_ws, cam_const(cam), view_in(grad_out), C, (int)mode, d_grad_in,
                                                                (long long)C * Hin * Win, Hin * Win, Hin, Win);
    else
        warp_backward_ordered_kernel<false><<<grd, 256, 0, st>>>(d_params_ws, cam_const(cam), view_in(grad_out), C, (int)mode, d_grad_in,
                                                                 (long long)C * Hin * Win, Hin * Win, Hin, Win);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_rasterize_sparse_depth(const double* d_tracks, const int32_t* d_counts, int32_t B, int32_t N, int32_t cols,
                                double fc0, double fc1, double cc0, double cc1, int32_t H, int32_t W,
                                int32_t* d_winner_ws, float* d_depth, void* stream) {
    if (B < 0 || N < 0 || cols < 4 || H <= 0 || W <= 0) return fail(VIDC_ERR_INVALID_ARGUMENT, "bad rasterisation sizes (tracks need >= 4 columns)");
    if (B == 0) return VIDC_OK;
    if (!d_depth || !d_winner_ws || (N > 0 && !d_tracks)) return fail(VIDC_ERR_INVALID_ARGUMENT, "null rasterisation pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const long long total = (long long)B * H * W;
    VIDC_CUDA(cudaMemsetAsync(d_winner_ws, 0xff, sizeof(int32_t) * (size_t)total, st));     // -1 everywhere
    if (N > 0) {
        rasterize_index_kernel<<<dim3((N + 127) / 128, B), 128, 0, st>>>(d_tracks, d_counts, B, N, cols, fc0, fc1, cc0, cc1, H, W, d_winner_ws);
        VIDC_LAUNCH_CHECK();
    }
    rasterize_write_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_tracks, N, cols, (long long)H * W, d_winner_ws, d_depth, total);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_warp_rgb_sparse_depth(const vidc_camera* cam, const vidc_image* rgb, const double* d_tracks, const int32_t* d_counts,
                               int32_t N, int32_t cols, double fc0, double fc1, double cc0, double cc1,
                               const float* d_Ig, const float* d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                               vidc_frame_params* d_params_ws, float* d_H_out, const vidc_image* rgb_out,
                               const vidc_image* depth_out, uint8_t* d_mask_u8, uint32_t* d_coverage, void* stream) {
    VIDC_TRY(check_cam(cam));
    VIDC_TRY(check_image(rgb, "rgb", 3, 3));
    VIDC_TRY(check_image(depth_out, "depth_out", 1, 1));
    if (N < 0 || cols < 4) return fail(VIDC_ERR_INVALID_ARGUMENT, "tracks need >= 4 columns");
    if (N > SPARSE_MAX_POINTS) return fail(VIDC_ERR_INVALID_ARGUMENT, "at most %d points per frame (got %d): rasterise and use vidc_warp_rgbd", SPARSE_MAX_POINTS, N);
    if (depth_mode != VIDC_BILINEAR && depth_mode != VIDC_NEAREST) return fail(VIDC_ERR_INVALID_ARGUMENT, "unknown interp mode %d", (int)depth_mode);
    if (rgb->h != cam->H || rgb->w != cam->W) return fail(VIDC_ERR_INVALID_ARGUMENT, "the sparse-depth path needs the input at the canvas size %dx%d", cam->W, cam->H);
    if (depth_out->n != rgb->n || depth_out->h != cam->H || depth_out->w != cam->W || depth_out->sw != 1 || depth_out->sh != cam->W)
        return fail(VIDC_ERR_INVALID_ARGUMENT, "depth_out must be (%d,1,%d,%d) with contiguous rows", rgb->n, cam->H, cam->W);
    if (N > 0 && !d_tracks) return fail(VIDC_ERR_INVALID_ARGUMENT, "null tracks pointer");
    VIDC_TRY(warp_rgbd_impl(cam, rgb, nullptr, d_Ig, d_Ia, B_gravity, VIDC_BILINEAR, d_params_ws, d_H_out, rgb_out, nullptr, d_mask_u8,
                            d_coverage, depth_out, stream));
    if (rgb->n == 0 || N == 0) return VIDC_OK;
    SparseArgs sa;
    sa.prm = d_params_ws; sa.cam = cam_const(cam); sa.tracks = d_tracks; sa.counts = d_counts; sa.N = N; sa.cols = cols;
    sa.fc0 = fc0; sa.fc1 = fc1; sa.cc0 = cc0; sa.cc1 = cc1; sa.dep_o = depth_out->data; sa.depo_sn = depth_out->sn; sa.mode = (int)depth_mode;
    warp_sparse_depth_kernel<<<dim3(rgb->n, 4), 256, 0, (cudaStream_t)stream>>>(sa);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

int vidc_condition_gravity(const float* d_raw, int32_t B, int32_t rule, float* d_Ig, float* d_Ia, void* stream) {
    if (B < 0 || (rule != 0 && rule != 1)) return fail(VIDC_ERR_INVALID_ARGUMENT, "bad batch or rule");
    if (B == 0) return VIDC_OK;
    if (!d_raw || !d_Ig || !d_Ia) return fail(VIDC_ERR_INVALID_ARGUMENT, "null gravity pointer");
    condition_gravity_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(d_raw, B, rule, d_Ig, d_Ia);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

#ifdef VIDC_BOX_TIMING
int vidc_debug_box_timing(unsigned long long* h_out8, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(h_out8, g_box_timing, sizeof(unsigned long long) * 8);
    if (reset) { unsigned long long z[8] = {0}; cudaMemcpyToSymbol(g_box_timing, z, sizeof z); }
    return VIDC_OK;
}
#endif

/* Test hook (tests/test_gpu_math.py): evaluates the kernels' shared-reciprocal divisions and the
   compiler's IEEE division on n operand triples.  d_out: 4*n floats. */
int vidc_debug_div(const float* d_u, const float* d_v, const float* d_s, int64_t n, float* d_out, void* stream) {
    if (n <= 0) return VIDC_OK;
    debug_div_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_u, d_v, d_s, n, d_out);
    VIDC_LAUNCH_CHECK();
    return VIDC_OK;
}

}  // extern "C"
