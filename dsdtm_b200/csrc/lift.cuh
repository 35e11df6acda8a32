// lift.cuh -- the per-feature arithmetic of Tracking::CraeteKeyframe (ref: src/Tracking.cpp:412-464), shared by keyframe_lift_kernel
// (ingest.cu, one frame from the host) and keyframe_lift_batch_kernel (keyframe.cu, the batched chain): one source, the same bits.
//   Frame::UndistortFeatures (ref: src/Frame.cpp:94-150) = cv::undistortPoints(K, dist, P = K), 5 fixed-point iterations in fp64,
//                            float in / float out, then mNormal = normalize(Pixel2Camera(px, 1.0)) (float evaluation, Q8)
//   Frame::Get_FeatureDetph  (ref: src/Frame.cpp:200-224): cvRound, centre + 4-neighbourhood
//   Frame::UnProject         (ref: src/Frame.cpp:152-157): T_c2w^-1 * Pixel2Camera(px, d)
// The raw 16-bit depth stays in HBM and is converted at the (<= 5) pixels a feature touches: float(u16) * float(1/scale) is the single
// rounding cv::Mat::convertTo performs, so the values are the ones the reference reads from its CV_32F image.
// fp64 non-contracted in OpenCV's / the reference's operation order: the undistorted pixels are bit-equal to cv2 4.13
// (tests/golden/undistort_cv2.npz through the oracle).
#pragma once

#include "ctx.cuh"
#include "se3_exact.cuh"

namespace dsdtm {

struct LiftCam {
    int w, h;
    float fx, fy, cx, cy;
    float dist[5];
    float inv_scale;
};

__device__ __forceinline__ float lift_depth_at(const LiftCam& a, const uint16_t* depth, int x, int y)
{
    if (x < 0 || y < 0 || x >= a.w || y >= a.h) return 0.f;      // the reference reads out of bounds here (undefined); we say 0
    return __fmul_rn((float)depth[(size_t)y * a.w + x], a.inv_scale);
}

// one feature that is not mbInitial; depth = the frame's raw depth or null (DSDTM_LIFT_NO_DEPTH); inv = T_c2w^-1
__device__ __forceinline__ dsdtm_lifted lift_feature(const LiftCam& a, const uint16_t* depth, const double* inv, float px_x, float px_y)
{
    dsdtm_lifted o;
    o.normal[0] = o.normal[1] = o.normal[2] = 0.0; o.point_w[0] = o.point_w[1] = o.point_w[2] = 0.0;
    // ---- cv::undistortPoints, K / dist CV_32F widened (ref: src/Camera.cpp:53-68), R = none, P = K, 5 iterations
    const double fx = (double)a.fx, fy = (double)a.fy, cx = (double)a.cx, cy = (double)a.cy;
    const double ifx = __ddiv_rn(1.0, fx), ify = __ddiv_rn(1.0, fy);
    const double k0 = (double)a.dist[0], k1 = (double)a.dist[1], p1 = (double)a.dist[2], p2 = (double)a.dist[3], k2 = (double)a.dist[4];
    const double u = (double)px_x, v = (double)px_y;
    double x = __dmul_rn(__dsub_rn(u, cx), ifx), y = __dmul_rn(__dsub_rn(v, cy), ify);
    const double x0 = x, y0 = y;
#pragma unroll 1
    for (int j = 0; j < 5; ++j) {
        const double xx = __dmul_rn(x, x), yy = __dmul_rn(y, y), r2 = __dadd_rn(xx, yy);
        const double den = __dadd_rn(1.0, __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(k2, r2), k1), r2), k0), r2));
        const double icdist = __ddiv_rn(1.0, den);                                  // numerator 1 + ((0*r2+0)*r2+0)*r2 == 1
        if (icdist < 0) { x = __dmul_rn(__dsub_rn(u, cx), ifx); y = __dmul_rn(__dsub_rn(v, cy), ify); break; }
        // deltaX = 2*p1*x*y + p2*(r2 + 2*x*x)   (left to right; the thin-prism terms are + 0)
        const double dX = __dadd_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, p1), x), y), __dmul_rn(p2, __dadd_rn(r2, __dmul_rn(__dmul_rn(2.0, x), x))));
        const double dY = __dadd_rn(__dmul_rn(p1, __dadd_rn(r2, __dmul_rn(__dmul_rn(2.0, y), y))), __dmul_rn(__dmul_rn(__dmul_rn(2.0, p2), x), y));
        x = __dmul_rn(__dsub_rn(x0, dX), icdist);
        y = __dmul_rn(__dsub_rn(y0, dY), icdist);
    }
    // RR = K: xx = fx*x + 0*y + cx ; ww = 1/(0*x + 0*y + 1) = 1
    const float ux = __double2float_rn(__dadd_rn(__dmul_rn(fx, x), cx)), uy = __double2float_rn(__dadd_rn(__dmul_rn(fy, y), cy));
    o.px[0] = ux; o.px[1] = uy;
    // ---- mNormal = Pixel2Camera(px, 1.0).normalize()  (float evaluation, ref: src/Camera.cpp:173-178, src/Frame.cpp:146-147)
    feature_normal_exact(ux, uy, a.fx, a.fy, a.cx, a.cy, o.normal);
    o.status = DSDTM_LIFT_NO_DEPTH; o.depth = -1.0f;
    if (depth) {
        // ---- Get_FeatureDetph (ref: src/Frame.cpp:200-224)
        const int px = __float2int_rn(ux), py = __float2int_rn(uy);
        float d = lift_depth_at(a, depth, px, py);
        if (d == 0.f) {
            const int dx[4] = { -1, 0, 1, 0 }, dy[4] = { 0, -1, 0, 1 };
            d = -1.0f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float t = lift_depth_at(a, depth, px + dx[k], py + dy[k]);
                if (t != 0.f && d < 0.f) d = t;
            }
        }
        o.depth = d;
        if (!(d < 0.f)) {                                                         // ref: src/Tracking.cpp:436-437
            // ---- UnProject (ref: src/Frame.cpp:152-157)
            const double c0 = (double)__fdiv_rn(__fmul_rn(d, __fsub_rn(ux, a.cx)), a.fx), c1 = (double)__fdiv_rn(__fmul_rn(d, __fsub_rn(uy, a.cy)), a.fy), c2 = (double)d;
            double w0, w1, w2;
            qrot_exact(inv, c0, c1, c2, w0, w1, w2);
            o.point_w[0] = __dadd_rn(w0, inv[4]); o.point_w[1] = __dadd_rn(w1, inv[5]); o.point_w[2] = __dadd_rn(w2, inv[6]);
            o.status = DSDTM_LIFT_OK;
        }
    }
    return o;
}

inline LiftCam make_lift_cam(const dsdtm_ctx* c, const float dist[5], float depth_scale)
{
    LiftCam a;
    a.w = c->cam.width; a.h = c->cam.height;
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    for (int k = 0; k < 5; ++k) a.dist[k] = dist[k];
    a.inv_scale = (float)(double)(1.0f / depth_scale);
    return a;
}

}  // namespace dsdtm
