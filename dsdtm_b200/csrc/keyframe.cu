// keyframe.cu -- Tracking::CraeteKeyframe (ref: src/Tracking.cpp:412-464) behind the batched tracked-pose chain (dsdtm_batch_run
// flags | 8): the key frame the tracker would create from each pair's cur frame, without a host round trip.
//
//   keyframe_seed_kernel       : one CTA per pair. Frame::Set_ExistingFeatures (ref: src/Feature_detection.cpp:43-50) marks the grid
//                                cell int(px.y / (float)CellSize) * grid_cols + int(px.x / (float)CellSize) of every match; a linear
//                                index outside [0, n_cells) is skipped (the reference's vector operator[] is undefined there). The
//                                pair's mask circles for detect_select_kernel: SearchLocalPoints' filled circles of radius CellSize
//                                (ref: src/Feature_alignment.cpp:100-113) and Frame::Set_Mask's of radius Camera.Min_dist (ref:
//                                src/Frame.cpp:286-298; every match carries a map point), both at the match's float px. max_new =
//                                Max_fts - n_matches, 0 for a pair that is not wanted or not tracked (n_matches -1). The wanted pairs' rows of the occupancy grid and
//                                of the FAST cell keys are zeroed here, so every replay rewrites everything it reads (no memset nodes).
//   (fast_kernel on the cur slots, detect_select_kernel: Feature_detector::detect, fast.cu / detect_select.cu)
//   keyframe_lift_batch_kernel : grid (corner blocks, pair). The new corners are not mbInitial: Frame::UndistortFeatures,
//                                Get_FeatureDetph on the pair's depth slot and UnProject with the pose after PoseOptimization, through
//                                the per-feature body lift.cuh shares with keyframe_lift_kernel.
#include "lift.cuh"

namespace dsdtm {

namespace {

static const int kSeedThreads = 256;
static const int kLiftThreads = 128;

struct SeedArgs {
    const dsdtm_match* match; const int* n_match; const uint8_t* want;
    uint8_t* occupied; unsigned long long* cells; int n_cells, grid_cols;
    float cell_f; int cell_size, min_dist, max_fts;
    dsdtm_circle* circ; int* n_circ; int* max_new;
};

__global__ void __launch_bounds__(kSeedThreads) keyframe_seed_kernel(const SeedArgs a)
{
    const int pair = blockIdx.x, tid = threadIdx.x;
    if (!a.want[pair] || a.n_match[pair] < 0) {          // n_match -1: the store-backed frame overflowed its rows and was not tracked
        if (tid == 0) { a.n_circ[pair] = 0; a.max_new[pair] = 0; }
        return;
    }
    uint8_t* occ = a.occupied + (size_t)pair * a.n_cells;
    unsigned long long* K = a.cells + (size_t)pair * a.n_cells;
    for (int i = tid; i < a.n_cells; i += kSeedThreads) { occ[i] = 0; K[i] = 0ull; }
    __syncthreads();
    const int n = a.n_match[pair];
    const dsdtm_match* M = a.match + (size_t)pair * DSDTM_TRACK_MAX_MATCHES;
    dsdtm_circle* C = a.circ + (size_t)pair * 2 * DSDTM_TRACK_MAX_MATCHES;
    for (int m = tid; m < n; m += kSeedThreads) {
        const float x = M[m].px[0], y = M[m].px[1];
        const long long k = (long long)__float2int_rz(__fdiv_rn(y, a.cell_f)) * a.grid_cols + __float2int_rz(__fdiv_rn(x, a.cell_f));
        if (k >= 0 && k < a.n_cells) occ[k] = 1;
        C[2 * m] = dsdtm_circle{ { x, y }, a.cell_size, 0 };
        C[2 * m + 1] = dsdtm_circle{ { x, y }, a.min_dist, 0 };
    }
    if (tid == 0) { a.n_circ[pair] = 2 * n; a.max_new[pair] = a.max_fts - n; }
}

struct LiftBatchArgs {
    LiftCam cam;
    const uint16_t* depth; size_t depth_px; const int* depth_slot;
    const double* pose;                           // n_pairs x 7 T_c2w after PoseOptimization
    const dsdtm_corner* corners; const int* n_new; int stride;
    dsdtm_lifted* out;
};

__global__ void __launch_bounds__(kLiftThreads) keyframe_lift_batch_kernel(const LiftBatchArgs a)
{
    const int pair = blockIdx.y;
    const int n = a.n_new[pair];
    if ((int)blockIdx.x * kLiftThreads >= n) return;                                  // the whole block: no barrier is skipped
    __shared__ double s_inv[7];
    if (threadIdx.x == 0) se3_inv_exact(a.pose + 7 * (size_t)pair, s_inv);
    __syncthreads();
    const int i = blockIdx.x * kLiftThreads + threadIdx.x;
    if (i >= n) return;
    const dsdtm_corner c = a.corners[(size_t)pair * a.stride + i];
    const int ds = a.depth_slot[pair];
    const uint16_t* depth = ds >= 0 ? a.depth + (size_t)ds * a.depth_px : nullptr;
    a.out[(size_t)pair * a.stride + i] = lift_feature(a.cam, depth, s_inv, (float)c.x, (float)c.y);   // Feature(Point2f(x, y))
}

}  // namespace

cudaError_t launch_keyframe_seed(dsdtm_ctx* c, int n_pairs, int min_dist, int max_fts, cudaStream_t s)
{
    SeedArgs a;
    a.match = c->trk_match_d; a.n_match = c->trk_nobs_d; a.want = c->kf_want_d;
    a.occupied = c->occupied_d; a.cells = c->cells_d; a.n_cells = c->n_cells; a.grid_cols = c->grid_cols;
    a.cell_f = (float)c->prm.cell_size; a.cell_size = c->prm.cell_size; a.min_dist = min_dist; a.max_fts = max_fts;
    a.circ = c->kf_circ_d; a.n_circ = c->kf_ncirc_d; a.max_new = c->kf_max_new_d;
    keyframe_seed_kernel<<<n_pairs, kSeedThreads, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_keyframe_lift_batch(dsdtm_ctx* c, int n_pairs, int stride, const float dist[5], float depth_scale, cudaStream_t s)
{
    LiftBatchArgs a;
    a.cam = make_lift_cam(c, dist, depth_scale);
    a.depth = c->depth_d; a.depth_px = (size_t)c->cam.width * c->cam.height; a.depth_slot = c->kf_depth_slot_d;
    a.pose = c->trk_pose_out_d;
    a.corners = c->kf_corner_d; a.n_new = c->kf_nnew_d; a.stride = stride;
    a.out = c->kf_lifted_d;
    dim3 grid((stride + kLiftThreads - 1) / kLiftThreads, n_pairs);
    keyframe_lift_batch_kernel<<<grid, kLiftThreads, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace dsdtm
