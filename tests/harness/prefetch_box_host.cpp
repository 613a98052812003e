// Host build of the inverse warp's L2 prefetch box (csrc/frame_params.cuh: inv_prefetch_box), the same source the sheared
// inverse kernel compiles, with the frame parameters and division proof it reads.
#include "../../vi_depth_completion_b200/csrc/frame_params.cuh"
// boxes: (B, tiles_y, tiles_x, 4) {x0, y0, x1, y1} inclusive, {0, 0, -1, -1} where the function returns false; proven: (B);
// params: (B) frame parameters
extern "C" void host_inv_prefetch_boxes(const vidc_camera* cam, const float* Ig, const float* Ia, int B, int* boxes, unsigned char* proven,
                                        vidc_frame_params* params) {
    const int tx = (cam->W + 31) / 32, ty = (cam->H + 31) / 32;
    for (int i = 0; i < B; ++i) {
        vidc_frame_params p;
        memset(&p, 0, sizeof p);
        vidc::frame_params_from_gravity(*cam, Ig + 3 * i, Ia + 3 * i, p);
        proven[i] = vidc::inv_division_proven(p, *cam) ? 1 : 0;
        params[i] = p;
        for (int t = 0; t < tx * ty; ++t) {
            const int X0 = (t % tx) * 32, Y0 = (t / tx) * 32;
            const int X1 = X0 + 31 < cam->W - 1 ? X0 + 31 : cam->W - 1, Y1 = Y0 + 31 < cam->H - 1 ? Y0 + 31 : cam->H - 1;
            int* b = boxes + ((size_t)i * tx * ty + t) * 4;
            if (!vidc::inv_prefetch_box(p.H, p.px_min, p.py_min, p.kw, p.kh, cam->cx, cam->cy, cam->inv_half_w, cam->inv_half_h, cam->W,
                                        cam->H, X0, Y0, X1, Y1, b)) {
                b[0] = 0; b[1] = 0; b[2] = -1; b[3] = -1;
            }
        }
    }
}
