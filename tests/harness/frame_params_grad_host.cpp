// Host build of the adjoint of the per-frame parameter chain (csrc/frame_params_grad.cuh), the same source the per-frame
// kernel of vidc_frame_params_backward compiles.
#include "../../vi_depth_completion_b200/csrc/frame_params_grad.cuh"
// gparams: (B) gradients of the frame parameters, gH: (B,3,3) or NULL; gg, ga: (B,3)
extern "C" void host_frame_params_backward(const vidc_camera* cam, const float* Ig, const float* Ia, int B, const vidc_frame_params* gparams,
                                           const float* gH, float* gg, float* ga) {
    for (int i = 0; i < B; ++i)
        vidc::frame_params_from_gravity_backward(*cam, Ig + 3 * i, Ia + 3 * i, gparams[i], gH ? gH + 9 * i : nullptr, gg + 3 * i, ga + 3 * i);
}
