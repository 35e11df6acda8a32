// ingest.cu -- SURVEY 8f-3 / 8f-4: what Tracking does to a frame before and while it becomes a keyframe.
//
//   depth_convert_kernel : depthImg.convertTo(CV_32F, 1/scale) (ref: src/Tracking.cpp:56) for callers that want the float image.
//                          HBM-bound streaming: 2 B read + 4 B written per pixel, 8-byte loads / 16-byte stores, all coalesced.
//   keyframe_lift_kernel : one thread per new feature of Tracking::CraeteKeyframe (ref: src/Tracking.cpp:412-464): UndistortFeatures,
//                          Get_FeatureDetph and UnProject with the per-feature body of lift.cuh, which the batched chain's
//                          keyframe_lift_batch_kernel (keyframe.cu) shares.
#include "lift.cuh"

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
    LiftCam cam;
    double pose[7];             // T_c2w; its inverse is computed by thread 0 of every block (cheap, keeps it one launch)
    const float* px_in; const uint8_t* initial; int n;
    dsdtm_lifted* out;
};

__global__ void __launch_bounds__(128) keyframe_lift_kernel(const LiftArgs a)
{
    __shared__ double s_inv[7];
    if (threadIdx.x == 0) se3_inv_exact(a.pose, s_inv);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    if (a.initial && a.initial[i]) {                                                // ref: src/Frame.cpp:140-141, src/Tracking.cpp:427-433
        dsdtm_lifted o;
        o.px[0] = a.px_in[2 * i]; o.px[1] = a.px_in[2 * i + 1];
        o.depth = 0.f; o.status = DSDTM_LIFT_SKIPPED;
        o.normal[0] = o.normal[1] = o.normal[2] = 0.0; o.point_w[0] = o.point_w[1] = o.point_w[2] = 0.0;
        a.out[i] = o;
        return;
    }
    a.out[i] = lift_feature(a.cam, a.depth, s_inv, a.px_in[2 * i], a.px_in[2 * i + 1]);
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
    a.cam = make_lift_cam(c, dist, depth_scale);
    for (int k = 0; k < 7; ++k) a.pose[k] = pose_c2w[k];
    a.px_in = c->lift_px_d; a.initial = have_initial ? c->lift_initial_d : nullptr; a.n = n; a.out = c->lift_out_d;
    keyframe_lift_kernel<<<(n + 127) / 128, 128, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace dsdtm
