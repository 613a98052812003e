// frame_params_grad.cuh -- adjoint of the per-frame parameter chain (frame_params.cuh): gradients of the frame parameters
// -> gradients of I_g and I_a.  One thread per frame (vidc_frame_params_backward), also compiled on the host by the tests.
//
// The reference builds its parameters with differentiable torch ops (networks/warping_2dof_alignment.py:35-58, :125-143), so
// autograd carries a gradient of H, R, Hinv, the bounding box and the canvas scale back to I_g and I_a.  This restates that
// backward in fp64, in reverse order of the forward:
//   ikw = 1/kw, ikh = 1/kh                                      :142-143
//   kw, kh from w_max, h_max in the 4:3 branch the forward took  :135-140
//   w_max, h_max from px / py min and max over the four corners  :127-133
//   px_j = c0 / c2, py_j = c1 / c2, c = H (X_j, Y_j, 1)          :126
//   H = (K R) K^-1, Hinv = (K R^T) K^-1                          :55-57
//   R = (I + 2 q4 S) + 2 S S, S = [q / (2 q4)]x                 :51-54
//   q4 = cos(atan2(|q|, d) / 2)                                  :44-48
//   q = g x a, d = a . g                                         :41-43
// The values are recomputed in fp64 from I_g and I_a.  The discrete decisions -- which branch of the 4:3 fit, which corners
// attain each min / max -- are those of the fp32 forward (frame_params_from_gravity), i.e. of the parameters the kernels used.
// Non-smooth points follow torch's autograd of the reference's ops:
//   - min / max ties split the gradient evenly among the tied corners (torch's backward of a full reduction,
//     evenly_distribute_backward; the reference reduces a 1-D tensor of four corners -- an assumption taken from the oracle's
//     restatement, since the reference's executed sources are not part of this repository);
//   - Tensor.norm at |q| = 0 (g parallel to a) passes no gradient.
// Non-finite gravity gives whatever this arithmetic gives; each frame is computed alone, so it never reaches other frames.
#pragma once
#include "frame_params.cuh"

namespace vidc {

VIDC_HD bool same_or_nan(float u, float v) { return u == v || (u != u && v != v); }

// gp: dL/d(field) for each field of vidc_frame_params (H, R, Hinv, px_min, py_min, kw, kh, ikw, ikh, w_max, h_max; the others
// are ignored).  gH: optional extra dL/dH (the Cg_H_C every reference method returns), NULL = 0.  gg, ga: dL/dI_g, dL/dI_a.
VIDC_HD void frame_params_from_gravity_backward(const vidc_camera& cam, const float* g, const float* a, const vidc_frame_params& gp,
                                                const float* gH, float* gg, float* ga) {
    // ---- fp32 forward: the kernels' parameters, for the branch and the tie sets
    vidc_frame_params p;
    frame_params_from_gravity(cam, g, a, p);
    const float Wm = (float)(cam.W - 1), Hmm = (float)(cam.H - 1);
    const float cxs[4] = {0.0f, Wm, 0.0f, Wm};
    const float cys[4] = {0.0f, 0.0f, Hmm, Hmm};
    float px32[4], py32[4];
    for (int j = 0; j < 4; ++j) {
        const float c0 = dot3_021(p.H[0], p.H[1], p.H[2], cxs[j], cys[j], 1.0f);
        const float c1 = dot3_021(p.H[3], p.H[4], p.H[5], cxs[j], cys[j], 1.0f);
        const float c2 = dot3_021(p.H[6], p.H[7], p.H[8], cxs[j], cys[j], 1.0f);
        px32[j] = c0 / c2; py32[j] = c1 / c2;
    }
    const bool branch_w = p.w_max > (4.0f * p.h_max) / 3.0f;

    // ---- fp64 forward values
    const double G[3] = {g[0], g[1], g[2]}, A[3] = {a[0], a[1], a[2]};
    const double q[3] = {A[2] * G[1] - A[1] * G[2], A[0] * G[2] - A[2] * G[0], A[1] * G[0] - A[0] * G[1]};
    const double d = A[0] * G[0] + A[1] * G[1] + A[2] * G[2];
    const double n = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2]);
    const double th = atan2(n, d);
    const double q4 = cos(0.5 * th), t = 2.0 * q4;
    const double qh[3] = {q[0] / t, q[1] / t, q[2] / t};
    const double S[9] = {0.0, -qh[2], qh[1], qh[2], 0.0, -qh[0], -qh[1], qh[0], 0.0};
    double R[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            double ss = 0.0;
            for (int k = 0; k < 3; ++k) ss += S[3 * r + k] * S[3 * k + c];
            R[3 * r + c] = ((r == c) ? 1.0 : 0.0) + t * S[3 * r + c] + 2.0 * ss;
        }
    double K[9], Ki[9], KR[9], H[9];
    for (int k = 0; k < 9; ++k) { K[k] = cam.K[k]; Ki[k] = cam.Kinv[k]; }
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) KR[3 * r + c] = K[3 * r] * R[c] + K[3 * r + 1] * R[3 + c] + K[3 * r + 2] * R[6 + c];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) H[3 * r + c] = KR[3 * r] * Ki[c] + KR[3 * r + 1] * Ki[3 + c] + KR[3 * r + 2] * Ki[6 + c];
    double cc[4][3], px[4], py[4];
    for (int j = 0; j < 4; ++j) {
        for (int r = 0; r < 3; ++r) cc[j][r] = H[3 * r] * (double)cxs[j] + H[3 * r + 1] * (double)cys[j] + H[3 * r + 2];
        px[j] = cc[j][0] / cc[j][2]; py[j] = cc[j][1] / cc[j][2];
    }
    double pxmin = px[0], pxmax = px[0], pymin = py[0], pymax = py[0];
    for (int j = 1; j < 4; ++j) {
        pxmin = fmin(pxmin, px[j]); pxmax = fmax(pxmax, px[j]); pymin = fmin(pymin, py[j]); pymax = fmax(pymax, py[j]);
    }
    const double w_max = pxmax - pxmin, h_max = pymax - pymin, Wf = cam.W, Hf = cam.H;
    const double kw = branch_w ? Wf / w_max : Wf / ((4.0 * h_max) / 3.0);
    const double kh = branch_w ? Hf / ((3.0 * w_max) / 4.0) : Hf / h_max;

    // ---- backward
    double gkw = (double)gp.kw - (double)gp.ikw / (kw * kw);                       // ikw = 1 / kw
    double gkh = (double)gp.kh - (double)gp.ikh / (kh * kh);
    double gw = gp.w_max, gh = gp.h_max;
    if (branch_w) { gw -= gkw * kw / w_max + gkh * kh / w_max; }                   // kw = W / w, kh = 4 H / (3 w)
    else          { gh -= gkh * kh / h_max + gkw * kw / h_max; }                   // kh = H / h, kw = 3 W / (4 h)
    const double g_pxmax = gw, g_pxmin = (double)gp.px_min - gw, g_pymax = gh, g_pymin = (double)gp.py_min - gh;
    // tie sets of the fp32 forward (torch.max / min propagate NaN: a NaN corner is "equal" to a NaN result)
    const float mx32 = tmax(tmax(tmax(px32[0], px32[1]), px32[2]), px32[3]), mn32 = tmin(tmin(tmin(px32[0], px32[1]), px32[2]), px32[3]);
    const float my32 = tmax(tmax(tmax(py32[0], py32[1]), py32[2]), py32[3]), ny32 = tmin(tmin(tmin(py32[0], py32[1]), py32[2]), py32[3]);
    int n_xmax = 0, n_xmin = 0, n_ymax = 0, n_ymin = 0;
    for (int j = 0; j < 4; ++j) {
        n_xmax += same_or_nan(px32[j], mx32); n_xmin += same_or_nan(px32[j], mn32); n_ymax += same_or_nan(py32[j], my32); n_ymin += same_or_nan(py32[j], ny32);
    }
    double gHt[9];
    for (int k = 0; k < 9; ++k) gHt[k] = (double)gp.H[k] + (gH ? (double)gH[k] : 0.0);
    for (int j = 0; j < 4; ++j) {
        double gpx = 0.0, gpy = 0.0;
        if (same_or_nan(px32[j], mx32)) gpx += g_pxmax / n_xmax;
        if (same_or_nan(px32[j], mn32)) gpx += g_pxmin / n_xmin;
        if (same_or_nan(py32[j], my32)) gpy += g_pymax / n_ymax;
        if (same_or_nan(py32[j], ny32)) gpy += g_pymin / n_ymin;
        if (gpx == 0.0 && gpy == 0.0) continue;
        const double gc[3] = {gpx / cc[j][2], gpy / cc[j][2], -(gpx * px[j] + gpy * py[j]) / cc[j][2]};
        for (int r = 0; r < 3; ++r) {
            gHt[3 * r] += gc[r] * (double)cxs[j];
            gHt[3 * r + 1] += gc[r] * (double)cys[j];
            gHt[3 * r + 2] += gc[r];
        }
    }
    // H = (K R) Ki, Hinv = (K R^T) Ki:  dR = K^T dH Ki^T,  d(R^T) = K^T dHinv Ki^T
    double gR[9];
    for (int k = 0; k < 9; ++k) gR[k] = gp.R[k];
    double tH[9], tHi[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            double s1 = 0.0, s2 = 0.0;
            for (int k = 0; k < 3; ++k) { s1 += gHt[3 * r + k] * Ki[3 * c + k]; s2 += (double)gp.Hinv[3 * r + k] * Ki[3 * c + k]; }
            tH[3 * r + c] = s1; tHi[3 * r + c] = s2;
        }
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            double s1 = 0.0, s2 = 0.0;
            for (int k = 0; k < 3; ++k) { s1 += K[3 * k + r] * tH[3 * k + c]; s2 += K[3 * k + r] * tHi[3 * k + c]; }
            gR[3 * r + c] += s1;
            gR[3 * c + r] += s2;
        }
    // R = I + t S + 2 S S:  dt = <dR, S>,  dS = t dR + 2 (dR S^T + S^T dR)
    double gt = 0.0, gS[9];
    for (int k = 0; k < 9; ++k) gt += gR[k] * S[k];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
            double s = 0.0;
            for (int k = 0; k < 3; ++k) s += gR[3 * r + k] * S[3 * c + k] + S[3 * k + r] * gR[3 * k + c];
            gS[3 * r + c] = t * gR[3 * r + c] + 2.0 * s;
        }
    const double gqh[3] = {gS[7] - gS[5], gS[2] - gS[6], gS[3] - gS[1]};
    double gq[3] = {gqh[0] / t, gqh[1] / t, gqh[2] / t};                           // qh = q / t
    gt -= (gqh[0] * qh[0] + gqh[1] * qh[1] + gqh[2] * qh[2]) / t;
    const double gq4 = 2.0 * gt;
    const double gth = -0.5 * sin(0.5 * th) * gq4;
    const double den = n * n + d * d;                                               // atan2(n, d)
    const double gn = gth * d / den, gd = -gth * n / den;
    if (n != 0.0)
        for (int k = 0; k < 3; ++k) gq[k] += gn * q[k] / n;                          // torch's norm backward: 0 at n = 0
    // q = g x a:  dg = a x dq,  da = dq x g;  d = a . g
    gg[0] = (float)(A[1] * gq[2] - A[2] * gq[1] + gd * A[0]);
    gg[1] = (float)(A[2] * gq[0] - A[0] * gq[2] + gd * A[1]);
    gg[2] = (float)(A[0] * gq[1] - A[1] * gq[0] + gd * A[2]);
    ga[0] = (float)(gq[1] * G[2] - gq[2] * G[1] + gd * G[0]);
    ga[1] = (float)(gq[2] * G[0] - gq[0] * G[2] + gd * G[1]);
    ga[2] = (float)(gq[0] * G[1] - gq[1] * G[0] + gd * G[2]);
}

}  // namespace vidc
