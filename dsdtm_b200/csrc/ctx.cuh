// ctx.cuh -- context, HBM layout and launch plumbing shared by the sm_100a kernels.
//
// HBM layout (DESIGN.md "Data layout"):
//   frame pool   : max_frames slots of frame_stride bytes; a slot holds the whole pyramid, level l dense (stride ==
//                  width, exactly like cv::pyrDown outputs) at byte offset lvl_off[l] (16-byte aligned), followed by
//                  >= 64 zero bytes of padding so that 1-past-the-end reads of the reference (Q4) stay inside the slot.
//   cells        : max_batch * n_cells packed 64-bit keys (score bits << 32 | inverted raster order) for FAST atomicMax.
//   batch inputs : feats / centers / poses / patches staged contiguously per pair.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/dsdtm_gpu.h"

namespace dsdtm {

struct LevelGeom {
    int w[DSDTM_MAX_LEVELS];
    int h[DSDTM_MAX_LEVELS];
    unsigned off[DSDTM_MAX_LEVELS];  // byte offset inside a frame slot
    int levels;
    unsigned frame_stride;           // bytes per slot
};

struct StageTimer {
    static const int kMaxEv = 64;
    cudaEvent_t ev0[kMaxEv], ev1[kMaxEv];
    int stage[kMaxEv];
    int n = 0;
    float ms[DSDTM_STAGE_COUNT] = {};
    int launches[DSDTM_STAGE_COUNT] = {};
};

}  // namespace dsdtm

namespace dsdtm { static const int kMaxStepStreams = 8; }

struct dsdtm_ctx {
    int device = 0;
    int sm_count = 148;
    dsdtm_cam cam;
    dsdtm_params prm;
    dsdtm::LevelGeom geo;
    int grid_rows = 0, grid_cols = 0, n_cells = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream[2] = { nullptr, nullptr };
    cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
    cudaEvent_t ev_chunk[4] = { nullptr, nullptr, nullptr, nullptr };
    cudaEvent_t ev_up[8] = {}, ev_done[8] = {};   // dsdtm_pair_batch_e2e: upload / kernels-done of chunk k (created once)
    cudaStream_t step_stream[dsdtm::kMaxStepStreams] = {};
    cudaEvent_t ev_fork = nullptr, ev_join[dsdtm::kMaxStepStreams] = {};
    int step_chunks = 1;                         // dsdtm_batch_run: pairs split over this many concurrent streams
    std::string err;
    long long launches = 0;
    long long captures = 0;                      // CUDA graphs captured by dsdtm_batch_run (dsdtm_graph_captures)
    bool profiling = false;
    dsdtm::StageTimer timer;
    float last_run_ms = 0.f;
    int pyr_kernel = 0;                          // 0 = auto (strip kernel where eligible), 1 = always the shared-memory tile kernel
    int sa_variant = 0;                          // 0 = shared-memory recompute kernel, 1 = L2 workspace kernel
    double* sa_ws_d = nullptr;                   // max_batch * 48 * nf doubles (variant 1)
    int sa_ctas_per_sm[11] = {};                 // resident CTAs per SM of sparse_align_kernel<WPP> for this max_feats (occupancy API), index = WPP
    int sa_wpp_override = 0;                     // 0 = pick warps-per-pair from the batch size

    // device memory
    uint8_t* frames_d = nullptr;                 // frame pool
    unsigned long long* cells_d = nullptr;       // max_batch * n_cells keys
    uint8_t* occupied_d = nullptr;               // max_batch * n_cells
    uint8_t* scoremap_d = nullptr;               // 2 * w0*h0 (score, nonmax) parity helper
    int* fast_tiles_d = nullptr;                 // FAST tile table (level, tx, ty packed)
    int n_fast_tiles = 0;

    // batch staging (device)
    int* ref_slots_d = nullptr;
    int* cur_slots_d = nullptr;
    dsdtm_ref_feat* feats_d = nullptr;           // max_batch * max_feats
    int* n_feats_d = nullptr;
    double* centers_d = nullptr;                 // max_batch * 3
    double* poses_in_d = nullptr;                // max_batch * 7
    double* poses_ref_d = nullptr;               // max_batch * 7: reference-frame poses of the batched refinement chain
    dsdtm_reproj* pair_reproj_d = nullptr;       // max_batch * max_patches: per-candidate records of the batched chain
    double* poses_out_d = nullptr;               // max_batch * 7
    int* n_tracked_d = nullptr;
    dsdtm_iter_log* log_d = nullptr;             // max_batch * kLogCap
    int* n_log_d = nullptr;
    uint8_t* patches_d = nullptr;                // max_batch * max_patches * 100
    double* patch_px_in_d = nullptr;             // max_batch * max_patches * 2 (start positions, never written by kernels)
    double* patch_px_d = nullptr;                // max_batch * max_patches * 2 (refined positions)
    int* patch_level_d = nullptr;
    int* patch_slot_d = nullptr;
    uint8_t* patch_conv_d = nullptr;
    // warp affine staging
    double* wa_A_d = nullptr;
    float* wa_px_d = nullptr;
    int* wa_meta_d = nullptr;                    // 3 ints per candidate: slot, ref_level, search_level
    dsdtm_candidate* cand_d = nullptr;           // max_batch * max_patches candidates (fused pipeline)
    // local-map snapshots (f-1), grown on demand
    dsdtm_kf_view* lm_kfs_d = nullptr;   size_t lm_kfs_cap = 0;
    dsdtm_obs* lm_obs_d = nullptr;       size_t lm_obs_cap = 0;
    dsdtm_map_point* lm_pts_d = nullptr; size_t lm_pts_cap = 0;
    double* lm_pose_d = nullptr;                 // lm_kfs_cap * 7 : T_cur * T_kf^-1
    dsdtm_reproj* lm_reproj_d = nullptr;         // lm_pts_cap
    // keyframe ingest (f-3 / f-4), allocated on first use
    int depth_slots = 4;
    uint16_t* depth_d = nullptr;                 // depth_slots * w*h raw depth
    float* depth_f32_d = nullptr;                // depth_slots * w*h (only for dsdtm_depth_convert_f32)
    float* lift_px_d = nullptr;          size_t lift_cap = 0;
    uint8_t* lift_initial_d = nullptr;
    dsdtm_lifted* lift_out_d = nullptr;
    uint8_t* clahe_src_d = nullptr;      size_t clahe_cap = 0;       // raw images waiting for CLAHE (frames)
    uint8_t* clahe_lut_d = nullptr;      size_t clahe_lut_cap = 0;   // per frame tiles * 256 bytes
    // device-resident map table for the local-map selection (f-1, caller side), grown on demand
    dsdtm_map_kf* mt_kfs_d = nullptr;    size_t mt_kfs_cap = 0;  size_t mt_kfs_n = 0;
    double* mt_pts_d = nullptr;          size_t mt_pts_cap = 0;  size_t mt_pts_n = 0;     // 3 doubles per row
    uint8_t* mt_vis_d = nullptr;         size_t mt_vis_cap = 0;
    double* mt_dist_d = nullptr;         size_t mt_dist_cap = 0;
    // device-resident map store (dsdtm_store_*)
    dsdtm_store_kf* st_kfs_d = nullptr;      size_t st_kfs_cap = 0, st_kfs_n = 0;
    dsdtm_store_feat* st_feats_d = nullptr;  size_t st_feats_cap = 0, st_feats_n = 0;
    dsdtm_store_point* st_pts_d = nullptr;   size_t st_pts_cap = 0, st_pts_n = 0;
    int* st_found_d = nullptr;               size_t st_found_cap = 0;      // per point: MapPoint::mnFound (appended points start at 1)
    std::vector<int32_t> st_kf_nfeat;        // host mirror of every key-frame row's feat_count (reserved rows of dsdtm_batch_commit_store)
    std::vector<int32_t> st_kf_slot;         // host mirror of every key-frame row's slot (dsdtm_batch_advance refuses a cur slot the store names)
    unsigned long long* st_claim_d = nullptr; size_t st_claim_cap = 0;     // per point: (~epoch << 32 | order) of the first local key frame that lists it
    uint8_t* st_vis_d = nullptr;             size_t st_vis_cap = 0;
    double* st_dist_d = nullptr;             size_t st_dist_cap = 0;
    int* st_sel_d = nullptr;                 // [0] = n_local, [1..16] = local rows, [17] = n_cand
    dsdtm_store_cand* st_out_d = nullptr;    size_t st_out_cap = 0;
    unsigned st_epoch = 0;
    int st_max_feats = 0;                    // largest feat_count of any key frame (grid width of the candidate kernels)
    // pose refinement (f-2), grown on demand
    dsdtm_ba_obs* po_obs_d = nullptr;    size_t po_obs_cap = 0;      // n_frames * obs_stride records
    double* po_res_d = nullptr;          size_t po_res_cap = 0;      // residual norms, same indexing
    int* po_nobs_d = nullptr;            size_t po_nobs_cap = 0;
    double* po_pose_in_d = nullptr;      size_t po_pose_in_cap = 0;  // 7 per frame
    double* po_pose_out_d = nullptr;     size_t po_pose_out_cap = 0;
    dsdtm_ba_summary* po_sum_d = nullptr; size_t po_sum_cap = 0;
    int po_solo_max = -1;                        // frames up to which a CTA of eight warps owns a frame (-1: the SM count); 0 = always one warp per frame
    // selection + pose optimization behind the batched chain (dsdtm_batch_stage_track): allocated once at max_batch size, owned by the
    // captured step (dsdtm_pose_optimize_batch's po_* buffers may be reallocated between two replays)
    int* trk_found_d = nullptr;                  // max_batch * max_patches found counts
    dsdtm_match* trk_match_d = nullptr;          // max_batch * DSDTM_TRACK_MAX_MATCHES
    dsdtm_ba_obs* trk_obs_d = nullptr;           // max_batch * DSDTM_TRACK_MAX_MATCHES
    int* trk_nobs_d = nullptr;                   // max_batch: matches per pair
    double* trk_pose_in_d = nullptr;             // max_batch * 7: cur.Get_Pose() after Run
    double* trk_pose_out_d = nullptr;            // max_batch * 7: after PoseOptimization
    double* trk_res_d = nullptr;                 // max_batch * DSDTM_TRACK_MAX_MATCHES
    dsdtm_ba_summary* trk_sum_d = nullptr;       // max_batch
    // the key frame behind the tracked pose (dsdtm_batch_stage_keyframe): allocated once per context at max_batch size, like trk_*, because
    // the replayed step points at them (det_buf_d / det_mask_d are regrown by dsdtm_detect_batch); cells_d / occupied_d are shared and
    // rewritten by every replay
    dsdtm_circle* kf_circ_d = nullptr;           // max_batch * 2 * DSDTM_TRACK_MAX_MATCHES: CellSize and Min_dist circles per match
    int* kf_ncirc_d = nullptr;                   // max_batch
    int* kf_max_new_d = nullptr;                 // max_batch: Max_fts - n_matches, 0 when not wanted
    dsdtm_corner* kf_corner_d = nullptr;         // max_batch * DSDTM_MAX_FEATS_LIMIT (row stride: the staged max_fts)
    dsdtm_lifted* kf_lifted_d = nullptr;         // same indexing
    int* kf_nnew_d = nullptr;                    // max_batch
    uint8_t* kf_exact_d = nullptr;               // max_batch
    int* kf_depth_slot_d = nullptr;              // max_batch, -1 = no depth
    uint8_t* kf_want_d = nullptr;                // max_batch
    int* kf_rows_d = nullptr;                    // max_batch: the wanted pairs in index order (the rows of the FAST grid)
    // store-backed local maps of the batched chain (dsdtm_batch_stage_store): allocated once per context at max_batch size, like trk_*,
    // except the per-point found counts, which follow the point table (any store change drops the captured steps)
    dsdtm_store_cand* sb_rec_d = nullptr;        // max_batch * max_patches records (row stride: the staged cands_per_frame)
    int* sb_ncand_d = nullptr;                   // max_batch: true candidate count per frame
    int* sb_local_d = nullptr;                   // max_batch * 17: n_local, then the local key-frame rows in rank order
    double* sb_pose10_d = nullptr;               // max_batch * 10: prior pose {c2w[7], centre[3]} = T_c2r * T_ref
    int2* sb_range_d = nullptr;                  // max_batch key-frame row ranges [begin, end)
    int* sb_found_d = nullptr;           size_t sb_found_cap = 0;    // per store point row: MapPoint::mnFound
    // dsdtm_batch_commit_store's scratch, grown on demand (never captured): per-frame counts / outputs and one push link per new feature
    int* cm_d = nullptr;                 size_t cm_cap = 0;
    int* cm_push_d = nullptr;            size_t cm_push_cap = 0;
    int* adv_d = nullptr;                        // dsdtm_batch_advance: max_batch * 2 (next cur slot, DSDTM_ADV_* per frame), allocated on first use
    // key-frame detection (dsdtm_detect_batch), grown on demand
    uint8_t* det_mask_d = nullptr;       size_t det_mask_cap = 0;    // n * w*h mask images: allocated by the first call that passes masks
    uint8_t* det_buf_d = nullptr;        size_t det_buf_cap = 0;     // small inputs (max_new, n_circles, circles) | outputs, one copy each way

    // pinned host staging for small synchronous calls
    uint8_t* pinned = nullptr;
    size_t pinned_bytes = 0;
    uint8_t* stage_pin = nullptr;                // fixed pinned arena for the small synchronous calls (see Stager / Arena in capi.cu)
    uint8_t* stage_dev = nullptr;                // its device mirror

    // staged batch description
    struct {
        bool staged = false;
        int n_pairs = 0, feat_stride = 0, max_level = 0, min_level = 0, max_iters = 0;
        int patches_per_pair = 0, align_iters = 0;
        bool map_staged = false;                           // dsdtm_batch_stage_map: the refinement chain's inputs are on the device
        int map_ppp = 0, max_search_level = 0, map_align_iters = 0;
        bool track_staged = false;                         // dsdtm_batch_stage_track: selection + pose optimization buffers are ready
        int track_iters = 0;
        bool store_staged = false;                         // dsdtm_batch_stage_store: bits 1..3 run on the map store instead
        bool store_all_rows = false;                       // no ranges staged: every frame reads rows [0, key frames at capture)
        int store_max_local = 0, store_cpf = 0, store_range_max = 0, store_range_end = 0, store_n_found = 0;
        bool store_found_live = false;                     // dsdtm_batch_stage_track_live: the selection reads st_found_d
        int commit_flags = 0;                              // flags of the last store-mode run with bit 2 not yet committed, 0 = none
        int advance_flags = 0;                             // flags of the last committed run not yet advanced (dsdtm_batch_advance), 0 = none
        std::vector<int32_t> ref_h, cur_h;                 // host mirrors of ref_slots_d / cur_slots_d (dsdtm_batch_stage, dsdtm_batch_advance)
        std::vector<int32_t> nm_h;                         // n_matches of the committed run, read back by the commit (frames held on overflow)
        std::vector<int32_t> kf_depth_h;                   // the staged depth slots (host copy, dsdtm_batch_upload_step)
        bool kf_staged = false;                            // dsdtm_batch_stage_keyframe: the key-frame half is ready
        int kf_min_dist = 0, kf_max_fts = 0, kf_n_wanted = 0;
        float kf_thr = 0.f, kf_dist[5] = {}, kf_depth_scale = 1.f;
        std::vector<uint8_t> kf_want;                      // the staged want mask (host copy)
        cudaGraphExec_t graph[16] = {};                    // [flags & 15]
        int graph_key[16][8];
    } batch;
};

namespace dsdtm {

static const int kLogCap = 256;  // per-pair iteration-log capacity on the device

inline int fail(dsdtm_ctx* c, int code, const char* what, cudaError_t e = cudaSuccess)
{
    char buf[512];
    if (e != cudaSuccess) snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    else snprintf(buf, sizeof buf, "%s", what);
    c->err = buf;
    return code;
}

#define DSDTM_CUDA(ctx, call)                                                        \
    do {                                                                             \
        cudaError_t e__ = (call);                                                    \
        if (e__ != cudaSuccess) return dsdtm::fail((ctx), DSDTM_E_CUDA, #call, e__); \
    } while (0)

// ---- stage timing (CUDA events on ctx->stream) ----
void stage_begin(dsdtm_ctx* c, int stage);
void stage_end(dsdtm_ctx* c, int n_launches);
int  stage_collect(dsdtm_ctx* c);

// ---- kernel launchers (each returns cudaGetLastError()) ----
cudaError_t pyramid_init(dsdtm_ctx* c);
cudaError_t launch_pyramid(dsdtm_ctx* c, int first_slot, int n, cudaStream_t s);
cudaError_t launch_pyramid_slots(dsdtm_ctx* c, const int* slots_d, int n, cudaStream_t s);
// kernel launches of one launch_pyramid / launch_pyramid_slots call (at most levels - 1: small levels may share one launch)
int pyramid_launches(dsdtm_ctx* c);
cudaError_t launch_fast_cells(dsdtm_ctx* c, int first_slot, int n, int barrier, float seed_score, bool use_occupied,
                              cudaStream_t s);
cudaError_t launch_fast_score_map(dsdtm_ctx* c, int slot, int level, int barrier, cudaStream_t s);
cudaError_t launch_sparse_align(dsdtm_ctx* c, int n_pairs, int feat_stride, int max_level, int min_level, int max_iters,
                                bool want_log, cudaStream_t s, int pair0 = 0, int n_pairs_total = 0);
cudaError_t launch_align2d(dsdtm_ctx* c, int n_patches, int max_iters, cudaStream_t s, int patch0 = 0, const int* n_dev = nullptr, dsdtm_store_cand* store_out = nullptr);
cudaError_t launch_warp_affine(dsdtm_ctx* c, int n, uint8_t* out_d, cudaStream_t s, int i0 = 0, const int* n_dev = nullptr);
cudaError_t launch_candidate_prep(dsdtm_ctx* c, int n, int cur_slot, int max_search_level, cudaStream_t s, int i0 = 0, const int* cur_slots_d = nullptr, int ppp = 0);
cudaError_t launch_clahe(dsdtm_ctx* c, int first_slot, int n, double clip_limit, int tiles_x, int tiles_y, cudaStream_t s);
int clahe_max_tiles_x();
int clahe_rows_per_cta();
cudaError_t launch_depth_convert(dsdtm_ctx* c, int first_slot, int n, float depth_scale, cudaStream_t s);
cudaError_t launch_keyframe_lift(dsdtm_ctx* c, int depth_slot, const double pose_c2w[7], const float dist[5], float depth_scale,
                                 bool have_initial, int n, cudaStream_t s);
cudaError_t launch_local_map_finalize(dsdtm_ctx* c, int n_pts, cudaStream_t s, dsdtm_reproj* out_d = nullptr, int i0 = 0);
// batched chain (one-key-frame local map per pair = its reference frame): reproject / closest observation / gates for pairs [pair0, pair0 + n_pairs)
cudaError_t launch_pair_candidates(dsdtm_ctx* c, int pair0, int n_pairs, int feat_stride, int ppp, cudaStream_t s);
cudaError_t launch_local_map(dsdtm_ctx* c, const double pose_cur[7], const double cur_center[3], int n_kfs, int n_pts, cudaStream_t s,
                             const double* pose_dev = nullptr);
struct StoreTrackArgs {
    int cur_slot, n_kfs, max_local, cap;
    double pose_cur[7], cur_center[3];
    const double* pose_dev = nullptr;           // {pose_c2w[7], centre[3]} on the device: overrides the two above
    // or: compose them on the device from the sparse alignment's T_c2r and the reference pose, into pose10_out (overrides all three)
    const double* t_c2r_dev = nullptr; double pose_ref[7] = {1, 0, 0, 0, 0, 0, 0}; double* pose10_out = nullptr;
    int max_search_level = 0;
};
cudaError_t launch_store_link(dsdtm_ctx* c, int feat_begin, int n_feats, cudaStream_t s);
cudaError_t launch_store_track(dsdtm_ctx* c, const StoreTrackArgs& a, cudaStream_t s);
const int* store_count_dev(dsdtm_ctx* c);     // number of candidate records of the last launch_store_track, on the device
// the batched chain on the map store (dsdtm_batch_stage_store): per frame, one prelude CTA (pose, close test, ranking, first-listing-wins
// walk into the frame's records in `order`) and the candidate records + SolveAffineMatrix / GetBestSearchLevel of entries
// [f * cpf, f * cpf + cpf); range_len = the longest staged range, all_end = the range of frames without one
size_t store_batch_smem(const dsdtm_ctx* c, int range_len, int max_local);
cudaError_t store_batch_init(dsdtm_ctx* c);
cudaError_t launch_store_batch(dsdtm_ctx* c, int n_pairs, bool all_rows, int range_len, int max_local, int cpf, int max_search_level, cudaStream_t s);
cudaError_t launch_compose_pose(dsdtm_ctx* c, const double* t_c2r_d, const double pose_ref_c2w[7], double* out10_d, cudaStream_t s);
cudaError_t launch_close_keyframes(dsdtm_ctx* c, const double pose_cur[7], int n_kfs, cudaStream_t s);
cudaError_t pose_opt_init(dsdtm_ctx* c);
cudaError_t launch_pose_opt(dsdtm_ctx* c, int n_frames, int obs_stride, int max_obs, int max_iters, bool want_res, bool want_sum,
                            cudaStream_t s);
// the same solve on explicit device buffers (res / sum may be null)
struct PoseOptIo {
    const dsdtm_ba_obs* obs; const int* n_obs; const double* pose_in;
    double* pose_out; double* res; dsdtm_ba_summary* sum;
};
cudaError_t launch_pose_opt_io(dsdtm_ctx* c, const PoseOptIo& io, int n_frames, int obs_stride, int max_obs, int max_iters, cudaStream_t s);
// SearchLocalPoints' selection over the batched chain's records + the PoseOptimization inputs of every pair (select.cu)
cudaError_t launch_track_select(dsdtm_ctx* c, int n_pairs, int feat_stride, int ppp, cudaStream_t s);
// the same over the store-backed records (sb_rec_d, cpf per frame): found counts per point row (n_found of them; later rows count 1)
cudaError_t launch_track_select_store(dsdtm_ctx* c, int n_pairs, int cpf, const int* found_d, int n_found, cudaStream_t s);
// dsdtm_batch_commit_store (store_commit.cu): found counts, bad flags, key frames, new points and observation chains of the last
// store-mode step; four launches on the tables as they are sized now (the caller reserved the worst case)
struct StoreCommitArgs {
    float threshold; bool keyframes;
    const int* kf_rows_d;                       // reserved key-frame row per frame, or null (append)
    int* cnt_d; int* out_d; int* push_d;        // 3n, 5n + 4, one per new feature row
};
cudaError_t launch_store_commit(dsdtm_ctx* c, const StoreCommitArgs& a, cudaStream_t s);
// dsdtm_batch_advance (sequence_advance.cu): every frame's next reference frame from the committed step; adv_d = next cur slot and
// DSDTM_ADV_* per frame, decided on the host
cudaError_t launch_sequence_advance(dsdtm_ctx* c, const int* adv_d, bool keyframes, cudaStream_t s);
size_t track_select_smem(int ppp);             // dynamic shared memory of one selection CTA for ppp records per frame
int track_select_key_bits(const dsdtm_ctx* c, int ppp);   // bits of a selection key for this grid and ppp (must be <= 64)
cudaError_t track_select_init(dsdtm_ctx* c);
int track_select_max_radius();                 // largest Camera.CellSize the selection's circle table holds
// Feature_detector::detect's sort + mask-circle selection over the cell keys of the last launch_fast_cells (detect_select.cu)
cudaError_t launch_detect_select(dsdtm_ctx* c, int n, float seed, const uint8_t* masks_d, const dsdtm_circle* circles_d, int circle_stride,
                                 const int* n_circles_d, const int* max_new_d, dsdtm_corner* out_d, int out_stride, int* n_out_d,
                                 uint8_t* exact_d, cudaStream_t s);
bool detect_select_fits(const dsdtm_ctx* c, size_t max_smem);
// the key frame behind the batched chain (keyframe.cu, fast.cu): occupancy + circles + max_new per pair, FAST on the cur slots of the
// wanted pairs (rows_d: their indices; n = 0 launches nothing), and the lift of the new corners
cudaError_t launch_keyframe_seed(dsdtm_ctx* c, int n_pairs, int min_dist, int max_fts, cudaStream_t s);
cudaError_t launch_fast_cells_slots(dsdtm_ctx* c, const int* slots_d, const int* rows_d, int n, float seed_score, cudaStream_t s);
cudaError_t launch_keyframe_lift_batch(dsdtm_ctx* c, int n_pairs, int stride, const float dist[5], float depth_scale, cudaStream_t s);
int detect_select_max_radius();                // largest dsdtm_circle.radius (and Camera.CellSize) the span table holds
int sparse_align_smem_bytes(int nf_pad);
size_t sparse_align_ws_doubles(int max_feats);
cudaError_t sparse_align_init(dsdtm_ctx* c);

}  // namespace dsdtm
