/*
 * vidc_b200.h -- C ABI of the B200-native gravity warp / unwarp path.
 *
 * This is the drop-in boundary: a plain C interface (pointers, sizes, a CUDA stream handle;
 * no torch or C++ types) that replaces, call for call, the PyTorch implementation in
 * MARSLab-UMN/vi_depth_completion:
 *
 *     networks/warping_2dof_alignment.py   class Warping2DOFAlignment          (:5-310)
 *     networks/surface_normal.py           mask / pyramid masks / renormalise  (:150-156, :170)
 *     normal_utils.py                      masked angular statistics           (:7-34)
 *
 * Each entry point cites the reference lines it replaces.  The Python mirror of the reference
 * class (vi_depth_completion_b200/warping_2dof_alignment.py) binds these symbols with ctypes;
 * INTEGRATION.md shows the binding a reference maintainer adds.
 *
 * Conventions
 *   - All tensors are IEEE fp32 (the reference casts with .type(torch.float), :115-116).
 *   - Pointers named d_* are DEVICE pointers on the CUDA device that is current when the call
 *     is made; pointers named h_* are HOST pointers.  Nothing is ever written through an input.
 *   - Images are described by a vidc_image: logical NCHW shape plus element strides, so both
 *     contiguous NCHW and channels-last (NHWC) storage are consumed / produced without a copy.
 *   - Every device entry point is asynchronous: it enqueues kernels on `stream` (a cudaStream_t
 *     passed as void*; NULL = the legacy default stream) and returns without synchronising.
 *   - Return value: VIDC_OK (0) or a negative vidc_status.  vidc_last_error() gives the message
 *     for the calling thread.  No entry point aborts the process.
 *   - Results are bit-identical to the reference executed by its CPU backend (torch 2.11, MKL: the pinned
 *     oracle, see DESIGN.md) -- parameters, sampling grids, warped images, masks and rotated /
 *     renormalised normals.  The reference's CUDA backend differs from its own CPU backend by an ulp in a
 *     few homography entries and in about half of the sampling coordinates (cuBLAS accumulate orders that
 *     depend on the problem size; measured on the B200, DESIGN.md section 2), so against that backend these
 *     results are exactly as close as the reference's CPU results are -- tests/test_gpu_reference_cuda.py.
 */
#ifndef VIDC_B200_H
#define VIDC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VIDC_ABI_VERSION 3

typedef enum vidc_status {
    VIDC_OK = 0,
    VIDC_ERR_INVALID_ARGUMENT = -1, /* shape / stride / null-pointer / enum problems (torch RuntimeError) */
    VIDC_ERR_BATCH_MISMATCH = -2,   /* x.shape[0] != I_g.shape[0]  (reference: AssertionError, :123,:224) */
    VIDC_ERR_CUDA = -3,             /* a CUDA runtime call failed; message carries cudaGetErrorString */
    VIDC_ERR_NO_DEVICE = -4         /* no sm_100 device is current */
} vidc_status;

typedef enum vidc_interp {
    VIDC_BILINEAR = 0, /* interp_mode='bilinear' (:108) */
    VIDC_NEAREST = 1,  /* interp_mode='nearest'             */
    VIDC_BICUBIC = 2   /* interp_mode='bicubic' (valid in F.grid_sample, never used by the reference's callers):
                          vidc_warp_forward and vidc_warp_normals_forward only, generic kernel, no backward */
} vidc_interp;

/* Camera constants of Warping2DOFAlignment.__init__ (:6-24).  Plain host struct. */
typedef struct vidc_camera {
    int32_t W, H;        /* ceil(2cx), ceil(2cy)                                  :13-14 */
    float K[9];          /* intrinsics, fp64 -> fp32                              :15,:19 */
    float Kinv[9];       /* np.linalg.inv(K) in fp64 -> fp32                      :16,:20 */
    float cx, cy;        /* principal point rounded once to fp32                  :149-150 */
    float inv_half_w;    /* float(1. / (W / 2))                                   :149 */
    float inv_half_h;    /* float(1. / (H / 2))                                   :150 */
    float fx, fy;
} vidc_camera;

/* Per-frame parameters produced by _build_homography (:35-58) and the bounding-box / scale
   block that the reference repeats in every method (:125-140, :168-194, :226-240). 48 floats. */
typedef struct vidc_frame_params {
    float H[9];      /* Cg_H_C      = K R K^-1                    :55 */
    float R[9];      /* Cg_R_C                                    :53-54 */
    float Hinv[9];   /* Cg_H_C_inv  = K R^T K^-1                  :56-57 */
    float px_min, py_min;  /* :128,:130 */
    float kw, kh;          /* :135-140 */
    float ikw, ikh;        /* "1./kw", "1./kh"  :142-143 */
    float w_max, h_max;    /* :132-133 */
    float fwd_col_major;   /* 1.0 when canvas rows of the forward warp run along source columns (roll beyond ~76 deg): kernels take column-major tiles */
    float inv_col_major;   /* same for the inverse warp */
    float reserved[11];    /* [0..9]: bit t set = 32x32 canvas tile t (row-major, <= 320 tiles) certainly lies outside the source
                              footprint of the forward warp -- written by the forward entry points, zero from every other
                              producer; [10]: 1.0 when the shared-reciprocal division of the inverse warp is provably exact for
                              every pixel of the frame (written by the inverse entry points' per-frame kernel), else 0 */
} vidc_frame_params;

/* Logical (N, C, H, W) image batch with element strides.  N <= 65535 frames per call (they ride on gridDim.z); one
 * frame must span fewer than 2^31 elements.  Larger batches: call once per slice. */
typedef struct vidc_image {
    float *data;                 /* device pointer */
    int32_t n, c, h, w;
    int64_t sn, sc, sh, sw;      /* strides in elements */
} vidc_image;

/* ------------------------------------------------------------------------------------------ */

/* ABI version of the loaded library. */
int vidc_abi_version(void);

/* Message of the last failing call on this thread ("" if none). */
const char *vidc_last_error(void);

/* Replaces Warping2DOFAlignment.__init__ (:6-24).  Host only. */
int vidc_camera_init(double fx, double fy, double cx, double cy, vidc_camera *cam);

/* Bytes of device scratch every `d_params_ws` argument below must provide for a batch of B frames: the B vidc_frame_params
   blocks followed by the per-tile tables of the kernels (today: the footprint boxes of the inverse warp, 16 bytes per 32x32
   tile).  16-byte aligned, caller-owned, may be reused across calls on the same stream.  Host only; 0 for B <= 0.
   (The reference re-allocates its scratch in every call, :118-122; there is no counterpart.) */
size_t vidc_workspace_bytes(const vidc_camera *cam, int32_t B);

/* Dataset-side gravity conditioning on device (SURVEY.md section 8 row f1): raw IMU gravity (B,3) -> I_g, I_a.
   rule 0 = Azure / Demo loaders (dataset.py:334-345, :472-483: negate y and z; psi < 1e-4 or cos(pitch) > 0.707
            -> a = [0,1,0], else a = [0, cos(pitch), sin(pitch)]);
   rule 1 = ScanNet compute_alignment_tensor (dataset.py:45-55: psi < 1e-6 or cos(pitch) <= 0.3 -> a = g, else [0,1,0]). */
int vidc_condition_gravity(const float *d_raw, int32_t B, int32_t rule, float *d_Ig, float *d_Ia, void *stream);

/* Sparse-depth rasterisation on device (SURVEY.md section 8 row f2; dataset.py:496-510, :316-329): d_tracks is (B,N,cols>=4) fp64
   [id, x, y, z, ...] (np.loadtxt rows), d_counts (B) the valid rows per frame (NULL = N); the pixel is
   (int(fc1*y/z + cc1), int(fc0*x/z + cc0)) in fp64 and, as in the reference's sequential loop, the LAST point on a pixel wins.
   d_winner_ws: scratch of B*H*W int32; d_depth: (B,1,H,W) fp32 output. */
int vidc_rasterize_sparse_depth(const double *d_tracks, const int32_t *d_counts, int32_t B, int32_t N, int32_t cols,
                                double fc0, double fc1, double cc0, double cc1, int32_t H, int32_t W,
                                int32_t *d_winner_ws, float *d_depth, void *stream);

/* SURVEY.md section 8 row f2, second half: forward warp of RGB plus the SPARSE depth of the frame's KLT tracks without ever
   building the (mostly zero) depth image: the tracks are rasterised as dataset.py:496-510 does (see above) into an on-chip
   table and warped analytically; depth_out (B,1,H,W) is bit-identical to vidc_warp_rgbd over vidc_rasterize_sparse_depth's
   image, for depth_mode bilinear and nearest.  N <= 2048 points per frame; the input must have the canvas size.  Everything
   else as vidc_warp_rgbd (mask, coverage, d_H_out, workspace). */
int vidc_warp_rgb_sparse_depth(const vidc_camera *cam, const vidc_image *rgb, const double *d_tracks, const int32_t *d_counts,
                               int32_t N, int32_t cols, double fc0, double fc1, double cc0, double cc1,
                               const float *d_Ig, const float *d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                               vidc_frame_params *d_params_ws, float *d_H_out, const vidc_image *rgb_out,
                               const vidc_image *depth_out, uint8_t *d_mask_u8, uint32_t *d_coverage, void *stream);

/* Replaces _build_homography (:35-58) plus the per-frame bbox / scale block (:125-140).
   d_Ig, d_Ia: (B,3) contiguous.  d_params: B entries. One thread per frame, no host sync. */
int vidc_frame_params_compute(const vidc_camera *cam, const float *d_Ig, const float *d_Ia, int32_t B,
                              vidc_frame_params *d_params, void *stream);

/* Parameters computed ONCE for a batch and shared by the forward and the inverse entry points (the reference rebuilds them in
   every call, :124 and :225, from the same I_g / I_a): fills d_params_ws (vidc_workspace_bytes(cam, B) bytes) with everything
   vidc_warp_rgbd, vidc_warp_rgb_sparse_depth and vidc_unwarp_normals need -- frame parameters, the forward kernels' exterior-tile
   bitmap and prefetch boxes, the inverse kernels' division proof -- and, if d_H_out is not NULL, Cg_H_C (B,3,3).  Those entry
   points then take d_Ig = d_Ia = NULL: "d_params_ws is prepared" (same camera, same B, written earlier in stream order; the
   call does not launch a per-frame kernel and leaves d_params_ws untouched, so it may be shared by any number of calls). */
int vidc_frame_params_prepare(const vidc_camera *cam, const float *d_Ig, const float *d_Ia, int32_t B,
                              vidc_frame_params *d_params_ws, float *d_H_out, void *stream);

/* _build_homography's return tuple (:58): scatters params into three contiguous (B,3,3) tensors.
   Any of d_H, d_R, d_Hinv may be NULL. */
int vidc_build_homography(const vidc_camera *cam, const float *d_Ig, const float *d_Ia, int32_t B,
                          float *d_H, float *d_R, float *d_Hinv, void *stream);

/* Layouts and speed (results never depend on them): contiguous NCHW planes whose width is a multiple of 32 and 16-byte aligned
   outputs (and mask) run the sheared kernels with the TMA write-out (bulk tensor stores, one output tensor map per call);
   outputs a tensor map cannot describe take the same kernels' LSU write-out; three-channel channels-last images (element
   strides sc = 1, sw = 3, sh = 3 W, sn = 3 W H, input and output alike) have their own sheared kernels at about the planar speed;
   everything else -- other strides, other widths -- is accepted without a copy by the strided kernels (about half the speed). */

/* Replaces warp_with_gravity_center_aligned (:108-156): fused params + grid + grid_sample.
   x: (B,C,Hin,Win) any strides; y: (B,C,cam.H,cam.W).  d_H_out (B,3,3) may be NULL.
   d_params_ws: caller-owned scratch of vidc_workspace_bytes(cam, B) bytes (B vidc_frame_params first; may alias across calls). */
int vidc_warp_forward(const vidc_camera *cam, const vidc_image *x, const float *d_Ig, const float *d_Ia,
                      int32_t B_gravity, vidc_interp mode, vidc_frame_params *d_params_ws,
                      float *d_H_out, const vidc_image *y, void *stream);

/* Fused single-pass forward warp of RGB (3ch, bilinear) AND sparse depth (1ch, depth_mode),
   plus the validity mask of surface_normal.py:151 and per-frame coverage counts.
   rgb_out/depth_out as in vidc_warp_forward.  Optional outputs (NULL to skip):
     d_mask_u8   (B, cam.H, cam.W) uint8, 1 where (R+G)+B > float(1e-2)
     d_coverage  (B) uint32, number of mask pixels per frame (warp-shuffle + one atomic per CTA;
                 zeroed by the call)
   depth may be NULL (RGB only). */
int vidc_warp_rgbd(const vidc_camera *cam, const vidc_image *rgb, const vidc_image *depth,
                   const float *d_Ig, const float *d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                   vidc_frame_params *d_params_ws, float *d_H_out,
                   const vidc_image *rgb_out, const vidc_image *depth_out,
                   uint8_t *d_mask_u8, uint32_t *d_coverage, void *stream);

/* vidc_warp_rgbd with the RGB frames as the loader decodes them (dataset.py:468-471): d_rgb_hwc is (B, Hin, Win, 3) uint8,
   contiguous, at any byte alignment (the layout vidc_to_tensor_u8 takes).  Every other argument, check and status is
   vidc_warp_rgbd's, including depth = NULL, the optional mask and coverage, and d_Ig = d_Ia = NULL with a workspace from
   vidc_frame_params_prepare.  Outputs are bit-identical to vidc_to_tensor_u8 followed by vidc_warp_rgbd: each tap is
   converted to x / 255 before the unchanged interpolation, so the float copy of the frames is never written (RGB + depth +
   mask: 24 B/px of HBM traffic instead of 48 B/px for the two passes).  Frames of the canvas size with a canvas width that
   is a multiple of 32 run the sheared kernels; everything else takes the strided kernel. */
int vidc_warp_rgbd_u8(const vidc_camera *cam, const uint8_t *d_rgb_hwc, int32_t B, int32_t Hin, int32_t Win,
                      const vidc_image *depth, const float *d_Ig, const float *d_Ia, int32_t B_gravity,
                      vidc_interp depth_mode, vidc_frame_params *d_params_ws, float *d_H_out,
                      const vidc_image *rgb_out, const vidc_image *depth_out,
                      uint8_t *d_mask_u8, uint32_t *d_coverage, void *stream);

/* Packed variant of vidc_warp_rgbd for callers that hold RGB + depth interleaved: d_in is (B, Hin, Win, 4) fp32
   (channels-last, C = 4: R, G, B, depth), d_out is (B, cam.H, cam.W, 4); both contiguous and 16-byte aligned.
   Every bilinear tap is one 128-bit load and every pixel one 128-bit store.  Same results per channel. */
int vidc_warp_rgbd_packed(const vidc_camera *cam, const float *d_in, int32_t B, int32_t Hin, int32_t Win,
                          const float *d_Ig, const float *d_Ia, int32_t B_gravity, vidc_interp depth_mode,
                          vidc_frame_params *d_params_ws, float *d_H_out, float *d_out, uint8_t *d_mask_u8,
                          uint32_t *d_coverage, void *stream);

/* Replaces inverse_warp_normal_image_with_gravity_center_aligned (:216-255) and, when
   `normalize` != 0, also the caller's F.normalize(z, dim=1) (surface_normal.py:170) in the same
   pass: gather + R^T rotation (+ renormalise).  x, z: (B,3,cam.H,cam.W).
   d_valid_u8 (B,H,W), optional: 1 where the sample footprint touched the canvas. */
int vidc_unwarp_normals(const vidc_camera *cam, const vidc_image *x, const float *d_Ig, const float *d_Ia,
                        int32_t B_gravity, int32_t normalize, vidc_frame_params *d_params_ws,
                        float *d_H_out, const vidc_image *z, uint8_t *d_valid_u8, void *stream);

/* Backward of the two warps w.r.t. the sampled image (SURVEY.md section 8 row f4; in the reference this is torch autograd
   through F.grid_sample, :152 / :251, and the bmm at :253).  grad_out: (B,C,cam.H,cam.W), any strides.
   inverse == 0: backward of warp_with_gravity_center_aligned  -> d_grad_in (B,C,Hin,Win) contiguous, zeroed by the call;
   inverse != 0: backward of inverse_warp_normal_image_...     -> grad w.r.t. x (B,3,H,W): scatter of R * grad_out.
   Scatter-add with atomics (as ATen's CUDA backward): results agree with autograd to rounding, not bit-for-bit, and may differ
   in the last bits from run to run; vidc_warp_backward_ordered below is the deterministic variant. */
int vidc_warp_backward(const vidc_camera *cam, const vidc_image *grad_out, const float *d_Ig, const float *d_Ia,
                       int32_t B_gravity, int32_t inverse, vidc_interp mode, vidc_frame_params *d_params_ws,
                       float *d_grad_in, int32_t Hin, int32_t Win, void *stream);

/* The same backward with ONE fixed summation order, so the gradient is a pure function of the inputs (bit-reproducible from
   run to run, at any batch position, on any stream).  Same arguments, checks and result layout as vidc_warp_backward; every
   element of d_grad_in is written (no zeroing needed).  Order contract: each element of grad_in starts at +0 and receives, in
   output row-major order (Y, then X), the contribution of every output pixel that has it among its in-bounds taps: the
   product w_tap * g rounded, then added with a separate rounding (no FMA).  A pixel reaches an element through at most one
   tap (bilinear: nw, ne, sw, se; nearest: the rint tap with weight 1, contribution g itself).  Coordinates and weights are
   the forward warps' bits; a non-finite coordinate contributes nothing; inverse != 0 first rotates g <- R g (k-ascending FMA
   chain from +0).  This is the order of a serial scatter loop (tests/harness/backward_scatter.c).  A gather
   kernel, one CTA per 32x32 tile of grad_in: no global atomics. */
int vidc_warp_backward_ordered(const vidc_camera *cam, const vidc_image *grad_out, const float *d_Ig, const float *d_Ia,
                               int32_t B_gravity, int32_t inverse, vidc_interp mode, vidc_frame_params *d_params_ws,
                               float *d_grad_in, int32_t Hin, int32_t Win, void *stream);

/* Bytes of device scratch vidc_warp_backward_params needs for a batch of B frames: one slot of fp64 partial sums per 32x32 tile
   of the canvas and frame (176 bytes per tile).  Caller-owned, no alignment beyond 8 bytes, reusable in stream order.  Host only;
   0 for B <= 0.  Separate from vidc_workspace_bytes, which it does not change. */
size_t vidc_warp_backward_params_scratch_bytes(const vidc_camera *cam, int32_t B);

/* Backward of the two warps w.r.t. the per-frame parameters (in the reference: torch autograd through the sampling grid of
   F.grid_sample, :142-152 / :242-251, and through the bmm with R^T at :253).  x: the forward's input, (B,C,Hin,Win) any strides;
   grad_out: (B,C,cam.H,cam.W) any strides; the same checks as vidc_warp_backward.
   inverse == 0 (forward warp, any C, bilinear or nearest): d_grad_params[b] receives dL/dHinv, dL/dpx_min, dL/dpy_min, dL/dikw,
     dL/dikh in the fields of those names;
   inverse != 0 (inverse warp, C = 3, bilinear): dL/dH, dL/dR, dL/dpx_min, dL/dpy_min, dL/dkw, dL/dkh.
   Every other field is 0, and 'nearest' gives 0 everywhere (ATen's grid gradient of nearest sampling is zero).  Per pixel it
   takes ATen's grid_sampler_2d_backward grid gradient at the forward's coordinates (a non-finite coordinate contributes 0).
   Order contract: each 32x32 output tile sums its pixels' terms in fp64 (each thread its column's rows in order, then a fixed
   shuffle tree and the 8 warps in order) into its own slot of d_scratch (vidc_warp_backward_params_scratch_bytes); a second
   pass adds a frame's tiles in row-major tile order and rounds once to fp32.  No global atomics: bit-reproducible from run to
   run, at any batch position, on any stream. */
int vidc_warp_backward_params(const vidc_camera *cam, const vidc_image *x, const vidc_image *grad_out, const float *d_Ig,
                              const float *d_Ia, int32_t B_gravity, int32_t inverse, vidc_interp mode, vidc_frame_params *d_params_ws,
                              void *d_scratch, vidc_frame_params *d_grad_params, void *stream);

/* Backward of _build_homography (:35-58) and the per-frame bbox / scale block (:125-143): the gradients of the frame parameters
   (d_grad_params: B entries, dL/d(field) in each field's place; fwd_col_major, inv_col_major and reserved are ignored) plus an
   optional extra gradient of the returned Cg_H_C (d_grad_H, (B,3,3), NULL = 0) -> dL/dI_g and dL/dI_a ((B,3) each, written).
   One thread per frame, fp64 arithmetic from I_g / I_a; the 4:3 branch and the corners that attain each min / max are those of
   the fp32 forward, and ties split the gradient evenly (torch's backward of a full min / max).  Each frame depends on its own
   inputs only. */
int vidc_frame_params_backward(const vidc_camera *cam, const float *d_Ig, const float *d_Ia, int32_t B,
                               const vidc_frame_params *d_grad_params, const float *d_grad_H, float *d_grad_Ig, float *d_grad_Ia,
                               void *stream);

/* Replaces image_sampler_forward_inverse (:158-214) including the aspect guard (:178-187).
   d_Rt (B,3,3), d_grid / d_inv_grid (B,H,W,2) contiguous; any may be NULL. */
int vidc_sampler_forward_inverse(const vidc_camera *cam, const float *d_Ig, const float *d_Ia, int32_t B,
                                 vidc_frame_params *d_params_ws, float *d_Rt, float *d_grid,
                                 float *d_inv_grid, void *stream);

/* Replaces warp_normal_image_with_gravity_center_aligned (:258-290) as evidently intended
   (the reference method raises at :259): forward warp of a 3-channel normal image followed by
   the per-pixel rotation z = R y. */
int vidc_warp_normals_forward(const vidc_camera *cam, const vidc_image *x, const float *d_Ig, const float *d_Ia,
                              int32_t B_gravity, vidc_interp mode, vidc_frame_params *d_params_ws,
                              float *d_H_out, const vidc_image *z, void *stream);

/* Replaces warp_with_homography (:292-310): explicit homographies, NON-uniform kw/kh (:299-300).
   d_Hm: (B,3,3) device.  The inverse is taken per frame in fp64 (np.linalg.inv, :301). */
int vidc_warp_with_homography(const vidc_camera *cam, const vidc_image *x, const float *d_Hm, int32_t B_h,
                              vidc_frame_params *d_params_ws, const vidc_image *y, void *stream);

/* surface_normal.py:151: mask = (x1[:,0]+x1[:,1])+x1[:,2] > float(1e-2), as uint8 and/or float. */
int vidc_validity_mask(const vidc_image *x1, uint8_t *d_mask_u8, float *d_mask_f32,
                       uint32_t *d_coverage, void *stream);

/* surface_normal.py:153-156: F.interpolate(mask, size, 'nearest') for float masks (B,1,Hin,Win). */
int vidc_mask_nearest(const float *d_mask, int32_t B, int32_t Hin, int32_t Win,
                      int32_t Hout, int32_t Wout, float *d_out, void *stream);

/* surface_normal.py:153-156, all levels in ONE launch (SURVEY.md section 8 row f3): source mask either uint8 (as written by
   vidc_warp_rgbd) or float; sizes_hw = {H0, W0, H1, W1, ...} (host array, 1..4 levels); d_outs = host array of `levels`
   device pointers to float (B,1,Hl,Wl) outputs. */
int vidc_mask_pyramid(const uint8_t *d_mask_u8, const float *d_mask_f32, int32_t B, int32_t Hin, int32_t Win,
                      int32_t levels, const int32_t *sizes_hw, float *const *d_outs, void *stream);

/* surface_normal.py:170: F.normalize(z, dim=1) for 3-channel images. */
int vidc_normalize3(const vidc_image *z, const vidc_image *out, void *stream);

/* normal_utils.py:20-34 (and :7-17): one pass producing, in d_out[4] (fp64, zeroed by the call):
     [0] sum(angle_deg * mask)   [1] sum(mask)   [2] sum |n*mask - gt*mask|   [3] sum cos_sim
   pred: (B,>=3,H,W) (first three channels used), gt: (B,3,H,W), mask: (B,1,H,W) float. */
int vidc_normal_stats(const vidc_image *gt, const vidc_image *pred, const vidc_image *mask,
                      int32_t normalize_prediction, double *d_out, void *stream);

/* Backward of the losses of normal_utils.py:7-34 w.r.t. pred_normals -- the reference back-propagates angle_L1 at
   network_run.py:186,248.  loss_mode: 0 = compute_normal_vectors_loss_l1(normalize_prediction=True), 1 = the same with
   normalize_prediction=False, 2 = compute_normal_vectors_loss_l2 (cosine).  d_stats = the four sums vidc_normal_stats
   produced for the same tensors ([1] = sum(mask) is read), d_grad_loss = the upstream gradient of the scalar loss (one
   float on the device, so nothing synchronises), grad_pred: (B,C,H,W) like pred, fully written (channels >= 3 get zeros). */
int vidc_normal_loss_backward(const vidc_image *gt, const vidc_image *pred, const vidc_image *mask, int32_t loss_mode,
                              const double *d_stats, const float *d_grad_loss, const vidc_image *grad_pred, void *stream);

/* ---- host-buffer end-to-end entry point (bench.py `e2e`, simple embedders) ------------------
   One frame batch through the whole path with HOST buffers: H2D of rgb/depth/normals/gravity,
   warp_rgbd, unwarp_normals(normalize=1), D2H of the four outputs.  Buffers are contiguous NCHW.
   Any of the output pointers may be NULL (not copied back).  Pinned host memory makes the copies
   asynchronous; the call synchronises `stream` before returning.  Device scratch is cached per
   (device, size) inside the library and released by vidc_release_workspace(). */
int vidc_warp_unwarp_host(const vidc_camera *cam, int32_t B,
                          const float *h_rgb, const float *h_depth, const float *h_normals,
                          const float *h_Ig, const float *h_Ia,
                          float *h_rgb_w, float *h_depth_w, uint8_t *h_mask, float *h_normals_cam,
                          void *stream);
int vidc_release_workspace(void);

/* ---- the data format on the DataLoader side of the path (dataset.py:468-471) ----------------
   torchvision's ToTensor on device: (B,H,W,C) uint8 as PIL decodes it -> (B,C,H,W) float32 = x / 255, the correctly rounded
   fp32 quotient ToTensor's .div(255) produces (bit-identical); C in 1..4.  15 B/px of HBM traffic for RGB. */
int vidc_to_tensor_u8(const uint8_t *d_hwc, int32_t B, int32_t H, int32_t W, int32_t C, float *d_chw, void *stream);

/* vidc_warp_unwarp_host with the RGB frames as (B,H,W,3) uint8 HOST buffers (what the reference's loader holds before
   to_tensor): a quarter of the RGB bytes cross PCIe and vidc_to_tensor_u8 runs on the device inside the pipeline.  Outputs
   are bit-identical to vidc_warp_unwarp_host on ToTensor(h_rgb_u8). */
int vidc_warp_unwarp_host_u8(const vidc_camera *cam, int32_t B,
                             const uint8_t *h_rgb_u8, const float *h_depth, const float *h_normals,
                             const float *h_Ig, const float *h_Ia,
                             float *h_rgb_w, float *h_depth_w, uint8_t *h_mask, float *h_normals_cam,
                             void *stream);

/* Test hook: runs the kernels' shared-reciprocal division helpers next to the compiler's IEEE
   division on n device operand triples (u, v, s); d_out receives 4*n floats
   [u/s fast | v/s fast | u/s IEEE | v/s IEEE].  Used by tests/test_gpu_math.py only. */
int vidc_debug_div(const float *d_u, const float *d_v, const float *d_s, int64_t n, float *d_out, void *stream);

/* Number of kernel launches issued by this library since load (all threads). For bench.py's
   gpu_launches accounting. */
uint64_t vidc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VIDC_B200_H */
