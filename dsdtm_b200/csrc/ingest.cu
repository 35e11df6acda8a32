// ingest.cu -- SURVEY 8f-3 / 8f-4: what Tracking does to a frame before and while it becomes a keyframe.
//
//   depth_convert_kernel : depthImg.convertTo(CV_32F, 1/scale) (ref: src/Tracking.cpp:56) for callers that want the float image.
//                          HBM-bound streaming: 2 B read + 4 B written per pixel, 8-byte loads / 16-byte stores, all coalesced.
//   keyframe_lift_kernel : one thread per new feature of Tracking::CraeteKeyframe (ref: src/Tracking.cpp:412-464):
//                            Frame::UndistortFeatures  (ref: src/Frame.cpp:94-150) = cv::undistortPoints(K, dist, P = K),
//                                                      5 fixed-point iterations in fp64, float in / float out, then
//                                                      mNormal = normalize(Pixel2Camera(px, 1.0)) (float evaluation, Q8)
//                            Frame::Get_FeatureDetph   (ref: src/Frame.cpp:200-224): cvRound, centre + 4-neighbourhood
//                            Frame::UnProject          (ref: src/Frame.cpp:152-157): T_c2w^-1 * Pixel2Camera(px, d)
//                          The raw 16-bit depth stays in HBM and is converted at the (<= 5) pixels a feature touches:
//                          float(u16) * float(1/scale) is the single rounding cv::Mat::convertTo performs, so the values are
//                          the ones the reference reads from its CV_32F image without ever writing that image.
// fp64 non-contracted in OpenCV's / the reference's operation order: the undistorted pixels are bit-equal to cv2 4.13
// (tests/golden/undistort_cv2.npz through the oracle).
#include "ctx.cuh"
#include "se3_exact.cuh"

namespace dsdtm {

namespace {

// Each thread converts 2 x 4 pixels, blockDim apart: every warp instruction is one fully coalesced request (256 B loads,
// 512 B stores) and both loads are in flight before the first use (scripts/bw_probe.cu: 6.9 TB/s for this shape vs 5.7 TB/s
// for a 16-byte load followed by two 32-byte-strided stores).
__global__ void __launch_bounds__(256) depth_convert_kernel(const uint16_t* __restrict__ src, float* __restrict__ dst, size_t n4, size_t n, float a)
{
    const size_t i = (size_t)blockIdx.x * 512 + threadIdx.x;
    uint2 v[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) if (i + 256 * k < n4) v[k] = __ldg(reinterpret_cast<const uint2*>(src) + i + 256 * k);
#pragma unroll
    for (int k = 0; k < 2; ++k)
        if (i + 256 * k < n4)
            reinterpret_cast<float4*>(dst)[i + 256 * k] = make_float4(__fmul_rn((float)(v[k].x & 0xFFFFu), a), __fmul_rn((float)(v[k].x >> 16), a),
                                                                      __fmul_rn((float)(v[k].y & 0xFFFFu), a), __fmul_rn((float)(v[k].y >> 16), a));
    if (i == 0)
        for (size_t k = n4 * 4; k < n; ++k) dst[k] = __fmul_rn((float)src[k], a);      // < 4 tail pixels
}

__global__ void __launch_bounds__(256) depth_convert_scalar_kernel(const uint16_t* __restrict__ src, float* __restrict__ dst, size_t n, float a)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __fmul_rn((float)src[i], a);
}

struct LiftArgs {
    const uint16_t* depth;      // w*h raw depth of the frame, or nullptr
    int w, h;
    float fx, fy, cx, cy;
    float dist[5];
    float inv_scale;
    double pose[7];             // T_c2w; its inverse is computed by thread 0 of every block (cheap, keeps it one launch)
    const float* px_in; const uint8_t* initial; int n;
    dsdtm_lifted* out;
};

__device__ __forceinline__ float depth_at(const LiftArgs& a, int x, int y)
{
    if (x < 0 || y < 0 || x >= a.w || y >= a.h) return 0.f;      // the reference reads out of bounds here (undefined); we say 0
    return __fmul_rn((float)a.depth[(size_t)y * a.w + x], a.inv_scale);
}

__global__ void __launch_bounds__(128) keyframe_lift_kernel(const LiftArgs a)
{
    __shared__ double s_inv[7];
    if (threadIdx.x == 0) se3_inv_exact(a.pose, s_inv);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    dsdtm_lifted o;
    o.px[0] = a.px_in[2 * i]; o.px[1] = a.px_in[2 * i + 1];
    o.depth = 0.f; o.status = DSDTM_LIFT_SKIPPED;
    o.normal[0] = o.normal[1] = o.normal[2] = 0.0; o.point_w[0] = o.point_w[1] = o.point_w[2] = 0.0;
    if (a.initial && a.initial[i]) { a.out[i] = o; return; }                       // ref: src/Frame.cpp:140-141, src/Tracking.cpp:427-433
    // ---- cv::undistortPoints, K / dist CV_32F widened (ref: src/Camera.cpp:53-68), R = none, P = K, 5 iterations
    const double fx = (double)a.fx, fy = (double)a.fy, cx = (double)a.cx, cy = (double)a.cy;
    const double ifx = __ddiv_rn(1.0, fx), ify = __ddiv_rn(1.0, fy);
    const double k0 = (double)a.dist[0], k1 = (double)a.dist[1], p1 = (double)a.dist[2], p2 = (double)a.dist[3], k2 = (double)a.dist[4];
    const double u = (double)o.px[0], v = (double)o.px[1];
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
    if (a.depth) {
        // ---- Get_FeatureDetph (ref: src/Frame.cpp:200-224)
        const int px = __float2int_rn(ux), py = __float2int_rn(uy);
        float d = depth_at(a, px, py);
        if (d == 0.f) {
            const int dx[4] = { -1, 0, 1, 0 }, dy[4] = { 0, -1, 0, 1 };
            d = -1.0f;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float t = depth_at(a, px + dx[k], py + dy[k]);
                if (t != 0.f && d < 0.f) d = t;
            }
        }
        o.depth = d;
        if (!(d < 0.f)) {                                                         // ref: src/Tracking.cpp:436-437
            // ---- UnProject (ref: src/Frame.cpp:152-157)
            const double c0 = (double)__fdiv_rn(__fmul_rn(d, __fsub_rn(ux, a.cx)), a.fx), c1 = (double)__fdiv_rn(__fmul_rn(d, __fsub_rn(uy, a.cy)), a.fy), c2 = (double)d;
            double w0, w1, w2;
            qrot_exact(s_inv, c0, c1, c2, w0, w1, w2);
            o.point_w[0] = __dadd_rn(w0, s_inv[4]); o.point_w[1] = __dadd_rn(w1, s_inv[5]); o.point_w[2] = __dadd_rn(w2, s_inv[6]);
            o.status = DSDTM_LIFT_OK;
        }
    }
    a.out[i] = o;
}

}  // namespace

cudaError_t launch_depth_convert(dsdtm_ctx* c, int first_slot, int n, float depth_scale, cudaStream_t s)
{
    const size_t px = (size_t)c->cam.width * c->cam.height;
    const size_t total = px * n;
    const float a = (float)(double)(1.0f / depth_scale);
    const uint16_t* src = c->depth_d + (size_t)first_slot * px;
    float* dst = c->depth_f32_d + (size_t)first_slot * px;
    if (px % 4 == 0) {                                      // slot offsets keep 8 / 16-byte alignment
        const size_t n4 = total / 4;
        depth_convert_kernel<<<(unsigned)((n4 + 511) / 512), 256, 0, s>>>(src, dst, n4, total, a);
    } else {
        depth_convert_scalar_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(src, dst, total, a);
    }
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_keyframe_lift(dsdtm_ctx* c, int depth_slot, const double pose_c2w[7], const float dist[5], float depth_scale,
                                 bool have_initial, int n, cudaStream_t s)
{
    LiftArgs a;
    const size_t px = (size_t)c->cam.width * c->cam.height;
    a.depth = depth_slot >= 0 ? c->depth_d + (size_t)depth_slot * px : nullptr;
    a.w = c->cam.width; a.h = c->cam.height;
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    for (int k = 0; k < 5; ++k) a.dist[k] = dist[k];
    a.inv_scale = (float)(double)(1.0f / depth_scale);
    for (int k = 0; k < 7; ++k) a.pose[k] = pose_c2w[k];
    a.px_in = c->lift_px_d; a.initial = have_initial ? c->lift_initial_d : nullptr; a.n = n; a.out = c->lift_out_d;
    keyframe_lift_kernel<<<(n + 127) / 128, 128, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace dsdtm
