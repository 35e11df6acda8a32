// pose_opt.cu -- Optimizer::PoseOptimization on the device (SURVEY 8f-2): one warp per frame, see pose_opt.cuh.
#include "ctx.cuh"
#include "pose_opt.cuh"

namespace dsdtm {

// Latency-bound by construction (a dependent chain of <= 100 LM iterations over a few hundred observations). Sweeps over many
// independent frames: one warp per frame, kSweepWarps frames per CTA, each warp in its own shared-memory slice -- the chip is
// filled by frames. A few frames (the per-frame call): one CTA of kSoloWarps warps per frame, so the pass over the observations
// is kSoloWarps times shorter. Both kernels are single instantiations: a frame's result does not depend on its neighbours.
#ifndef DSDTM_PO_SWEEP_WARPS
#define DSDTM_PO_SWEEP_WARPS 4
#endif
// DSDTM_PO_SWEEP_MINB: CTAs per SM the sweep kernel is compiled for (a register cap); measured in scripts/po_variants.sh:
// every cap spills and is slower than the uncapped 238 registers (0.674 ms per 4096 frames; 168 regs 0.739, 128 regs 0.818, 96 regs 0.926).
#ifdef DSDTM_PO_SWEEP_MINB
#define DSDTM_PO_SWEEP_BOUNDS __launch_bounds__(DSDTM_PO_SWEEP_WARPS * 32, DSDTM_PO_SWEEP_MINB)
#else
#define DSDTM_PO_SWEEP_BOUNDS __launch_bounds__(DSDTM_PO_SWEEP_WARPS * 32)
#endif
static const int kSweepWarps = DSDTM_PO_SWEEP_WARPS;
static const int kSoloWarps = 8;
static const int kPoseOptSmemLimit = 200 * 1024;

__global__ void DSDTM_PO_SWEEP_BOUNDS
pose_opt_sweep_kernel(int n_frames, const dsdtm_ba_obs* __restrict__ obs, int obs_stride, const int* __restrict__ n_obs,
                      const double* __restrict__ poses_in, int max_iters, double* __restrict__ poses_out,
                      double* __restrict__ res_norm, dsdtm_ba_summary* __restrict__ summaries, int soa_stride)
{
    extern __shared__ double po_smem[];
    const int warp = threadIdx.x >> 5;
    const int frame = blockIdx.x * (blockDim.x >> 5) + warp;
    if (frame >= n_frames) return;                 // whole warps leave together; no CTA-wide barrier follows
    WarpLanes ln;
    pose_optimize(ln, n_obs[frame], obs + (size_t)frame * obs_stride, po_smem + (size_t)warp * soa_stride,
                  poses_in + 7 * (size_t)frame, max_iters, poses_out + 7 * (size_t)frame,
                  res_norm ? res_norm + (size_t)frame * obs_stride : nullptr, summaries ? summaries + frame : nullptr);
}

__global__ void __launch_bounds__(kSoloWarps * 32, 1)
pose_opt_solo_kernel(const dsdtm_ba_obs* __restrict__ obs, int obs_stride, const int* __restrict__ n_obs,
                     const double* __restrict__ poses_in, int max_iters, double* __restrict__ poses_out,
                     double* __restrict__ res_norm, dsdtm_ba_summary* __restrict__ summaries)
{
    extern __shared__ double po_smem[];
    __shared__ double red[2 * kSoloWarps * 28];
    const int frame = blockIdx.x;
    CtaLanes<kSoloWarps, 28> ln(red);
    pose_optimize(ln, n_obs[frame], obs + (size_t)frame * obs_stride, po_smem, poses_in + 7 * (size_t)frame, max_iters,
                  poses_out + 7 * (size_t)frame, res_norm ? res_norm + (size_t)frame * obs_stride : nullptr,
                  summaries ? summaries + frame : nullptr);
}

cudaError_t pose_opt_init(dsdtm_ctx*)
{
    cudaError_t e = cudaFuncSetAttribute(pose_opt_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoseOptSmemLimit);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(pose_opt_solo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPoseOptSmemLimit);
}

// max_obs = an upper bound of the batch's n_obs (sizes the shared-memory slice of a frame: 48 bytes per observation; the slice is
// laid out by the frame's own n_obs, so the bound never changes a result)
cudaError_t launch_pose_opt_io(dsdtm_ctx* c, const PoseOptIo& io, int n_frames, int obs_stride, int max_obs, int max_iters, cudaStream_t s)
{
    const int soa_stride = 6 * ((max_obs + 1) & ~1);
    const size_t per_frame = (size_t)soa_stride * sizeof(double);
    const int solo_max = c->po_solo_max >= 0 ? c->po_solo_max : c->sm_count;   // one solo CTA per SM: 64 frames 108 us; two per SM (296 frames) 189 us vs 167 us for the sweep kernel
    if (n_frames <= solo_max) {
        pose_opt_solo_kernel<<<n_frames, kSoloWarps * 32, per_frame, s>>>(io.obs, obs_stride, io.n_obs, io.pose_in, max_iters, io.pose_out,
                                                                        io.res, io.sum);
    } else {
        int wpc = kSweepWarps;                     // frames per CTA, while their slices fit
        while (wpc > 1 && wpc * per_frame > (size_t)kPoseOptSmemLimit) wpc >>= 1;
        pose_opt_sweep_kernel<<<(n_frames + wpc - 1) / wpc, wpc * 32, wpc * per_frame, s>>>(n_frames, io.obs, obs_stride, io.n_obs,
                                                                                         io.pose_in, max_iters, io.pose_out, io.res, io.sum, soa_stride);
    }
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_pose_opt(dsdtm_ctx* c, int n_frames, int obs_stride, int max_obs, int max_iters, bool want_res, bool want_sum,
                            cudaStream_t s)
{
    const PoseOptIo io = { c->po_obs_d, c->po_nobs_d, c->po_pose_in_d, c->po_pose_out_d, want_res ? c->po_res_d : nullptr,
                           want_sum ? c->po_sum_d : nullptr };
    return launch_pose_opt_io(c, io, n_frames, obs_stride, max_obs, max_iters, s);
}

}  // namespace dsdtm
