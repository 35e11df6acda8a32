/*
 * dsdtm_gpu.h -- C-ABI of the B200-native tracking front end (drop-in boundary, SURVEY.md section 8b).
 *
 * The reference (gaochq/DSDTM) has no FFI: the seam is three C++ classes and one Frame method, all called
 * from the tracking thread. Each entry point below names the reference interface it replaces ("ref:" paths are
 * below the reference root). No C++ / torch type crosses this boundary: plain pointers, sizes, PODs.
 *
 * Conventions
 *   - every pointer is HOST memory unless the name ends in _d; pinned host memory makes copies asynchronous;
 *   - return 0 = ok, < 0 = error (DSDTM_E_*); never throws, never aborts; dsdtm_last_error() gives the text;
 *   - a context is single-thread-affine (one per host thread / per GPU), like the reference's tracking thread;
 *   - pose7 = {qw,qx,qy,qz,tx,ty,tz}: unit quaternion + translation = Sophus::SE3's state;
 *   - images are 8-bit gray, row-major, level images dense (stride == width) like cv::pyrDown outputs;
 *   - there is NO CPU fallback: without a CUDA device dsdtm_create() fails.
 */
#ifndef DSDTM_GPU_H
#define DSDTM_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DSDTM_ABI_VERSION 1
#define DSDTM_MAX_LEVELS 8
#define DSDTM_MAX_FEATS_LIMIT 512 /* hard upper bound for dsdtm_params.max_feats */
/* frames or frame pairs one batched call takes at most, whatever max_batch is: the pyramid, FAST, CLAHE and key-frame lift kernels
 * index the frame with gridDim.y / gridDim.z, which CUDA caps at 65535. A larger n is DSDTM_E_ARG with nothing enqueued. */
#define DSDTM_MAX_BATCH_FRAMES 65535

enum {
    DSDTM_OK = 0,
    DSDTM_E_ARG = -1,    /* bad argument */
    DSDTM_E_CUDA = -2,   /* CUDA runtime error (text in dsdtm_last_error) */
    DSDTM_E_NOMEM = -3,  /* device / pinned allocation failed */
    DSDTM_E_STATE = -4   /* call sequence error (e.g. batch not staged) */
};

typedef struct dsdtm_ctx dsdtm_ctx;

/* ref: include/Camera.h:137-163, src/Camera.cpp:34-48 -- intrinsics are float in the reference on purpose */
typedef struct {
    int   width, height;
    float fx, fy, cx, cy;
    float f; /* Camera.f: the focal length Sprase_ImgAlign's Jacobian uses (ref: src/Sprase_ImageAlign.cpp:70,160) */
} dsdtm_cam;

/* ref: Config keys read at src/Feature_detection.cpp:12-16, src/Feature_alignment.cpp:24-30, src/Frame.cpp:51-52 */
typedef struct {
    int levels;      /* Camera.MaxPyraLevels (1..DSDTM_MAX_LEVELS) */
    int cell_size;   /* Camera.CellSize */
    int max_feats;   /* capacity: reference features per frame pair handed to sparse alignment (<= 512) */
    int max_patches; /* capacity: Align2D patches per frame */
    int max_frames;  /* frame slots in the device pool (each holds one full pyramid) */
    int max_batch;   /* capacity: frame pairs per batched call. Not capped: it also sizes the patch capacity max_batch * max_patches,
                      * but a batched call of frames or pairs takes at most DSDTM_MAX_BATCH_FRAMES of them */
} dsdtm_params;

/* One reference feature as Sprase_ImgAlign::GetJocabianMat reads it (ref: src/Sprase_ImageAlign.cpp:84-103) */
typedef struct {
    float  px[2];      /* Feature::mpx       ref: include/Feature.h:19 */
    int    level;      /* Feature::mlevel    ref: include/Feature.h:20 */
    int    initial;    /* Feature::mbInitial ref: include/Feature.h:23 */
    double normal[3];  /* Feature::mNormal   ref: include/Feature.h:24 */
    double point_w[3]; /* Feature::Mpt->Get_Pose() snapshot, ref: src/MapPoint.cpp:38-43 */
} dsdtm_ref_feat;      /* 64 bytes */

/* ref: include/Feature_detection.h:19-33 (struct Corner; angle is always 0 and dropped) */
typedef struct {
    int   x, y, level;
    float score;
} dsdtm_corner; /* 16 bytes */

/* One Gauss-Newton iteration of Sprase_ImgAlign::GaussNewtonSolver (ref: src/Sprase_ImageAlign.cpp:310-343) */
typedef struct {
    int    level, iter;
    int    n_pts;  /* visible features in this ComputeResiduals call */
    int    flags;  /* bit0 update accepted, bit1 reverted (chi2 increase / NaN), bit2 NaN solve, bit3 |x|<=1e-8 */
    double chi2;   /* chi2New = mean squared residual */
    double x[6];   /* GN step (upsilon, omega) */
} dsdtm_iter_log;  /* 72 bytes */

/* Per-stage device timing, filled when profiling is on (CUDA events on the context's stream). */
enum { DSDTM_STAGE_PYRAMID = 0, DSDTM_STAGE_FAST = 1, DSDTM_STAGE_SPARSE_ALIGN = 2, DSDTM_STAGE_ALIGN2D = 3,
       DSDTM_STAGE_WARP_AFFINE = 4, DSDTM_STAGE_CAND_PREP = 5, DSDTM_STAGE_LOCAL_MAP = 6, DSDTM_STAGE_INGEST = 7, DSDTM_STAGE_POSE_OPT = 8, DSDTM_STAGE_COUNT = 9 };

/* ---------------------------------------------------------------- context ---------------------------------- */
int         dsdtm_abi_version(void);
/* Creates a context on CUDA device `device`. Returns NULL on failure (call dsdtm_create_error() for the text). */
dsdtm_ctx*  dsdtm_create(int device, const dsdtm_cam* cam, const dsdtm_params* params);
const char* dsdtm_create_error(void);
void        dsdtm_destroy(dsdtm_ctx* ctx);
const char* dsdtm_last_error(const dsdtm_ctx* ctx);
int         dsdtm_sync(dsdtm_ctx* ctx);
/* level geometry of the device pyramid: width, height and byte offset of `level` inside a frame slot */
int         dsdtm_level_info(const dsdtm_ctx* ctx, int level, int* w, int* h, size_t* offset);
size_t      dsdtm_frame_stride(const dsdtm_ctx* ctx);
/* pinned host memory helpers (for asynchronous copies at the boundary) */
void*       dsdtm_host_alloc(size_t bytes);
void        dsdtm_host_free(void* p);
/* kernels launched by this context since creation (bench.py's gpu_launches) */
long long   dsdtm_launch_count(const dsdtm_ctx* ctx);
/* CUDA graphs dsdtm_batch_run has captured on this context since creation: a run that only replays a captured step adds nothing */
long long   dsdtm_graph_captures(const dsdtm_ctx* ctx);
/* measurement aid (no reference counterpart): the DFMA throughput this GPU sustains on dependency-free streams, in TFLOP/s (2 flops
 * per DFMA) and in warp instructions per clock and SM at the nominal maximum clock -- the ceiling bench.py puts the fp64
 * sparse-alignment kernel against. Runs a ~10 ms kernel on the context's stream and synchronises. */
int         dsdtm_probe_fp64(dsdtm_ctx* ctx, double* tflops, double* dfma_warp_insts_per_clk_per_sm);
/* tuning knobs (never change results): "sa_warps_per_pair" = 0 (auto: 10 for a lone pair, 4, or 3 from four pairs per SM
 * upwards) | 1 | 2 | 3 | 4 | 5 | 10 warps of one CTA per frame pair;
 * "pyramid_kernel" = 0 (auto: TMA bulk-staged kernel where the level shape allows, whole-level kernel for the ragged tail, tile
 * kernel otherwise) | 1 (shared-memory tile kernel everywhere) | 2 (register / DP4A strip kernel, the round-1 default);
 * "sa_variant" = 0 (shared-memory recompute kernel) | 1 (L2 workspace kernel); "step_chunks" = 1..8 concurrent streams
 * over which dsdtm_batch_run splits the ALIGNMENT stages of a step (all pyramids of the step are built first on the origin
 * stream, so a ref slot may be another pair's cur slot, as in the unchunked order); "depth_slots" = size of the depth
 * pool (before its first use); "pose_opt_solo_max" = frames per dsdtm_pose_optimize_batch call up to which a CTA of eight warps
 * owns a frame (-1 = the SM count, 0 = always one warp per frame; the two kernels agree to rounding, not bitwise) */
int         dsdtm_set_option(dsdtm_ctx* ctx, const char* key, int value);
/* stage profiling: on != 0 brackets every stage with CUDA events; get returns accumulated ms and launch counts */
int         dsdtm_profile(dsdtm_ctx* ctx, int on);
int         dsdtm_profile_get(dsdtm_ctx* ctx, float ms[DSDTM_STAGE_COUNT], int launches[DSDTM_STAGE_COUNT], int reset);

/* ---------------------------------------------------------------- (a) image pyramid ------------------------ */
/* replaces Frame::ComputeImagePyramid (ref: src/Frame.cpp:74-81; include/Frame.h:32): uploads level 0 and builds
 * levels 1..levels-1 with cv::pyrDown semantics into frame slot `slot`. stride = bytes per input row. */
int dsdtm_frame_upload_pyramid(dsdtm_ctx* ctx, int slot, const uint8_t* img, int stride);
/* same, and additionally returns the host copies of levels 1..levels-1 that Frame::mvImg_Pyr carries (ref: include/Frame.h
 * mvImg_Pyr) in the SAME synchronisation: levels_out receives dsdtm_frame_stride() - level-1-offset bytes laid out like the
 * slot (level l at dsdtm_level_info offset[l] - offset[1], dense rows). levels_out may be NULL. */
int dsdtm_frame_upload_pyramid_host(dsdtm_ctx* ctx, int slot, const uint8_t* img, int stride, uint8_t* levels_out);
/* dsdtm_frame_upload_pyramid without the closing synchronisation: the copy and the pyramid kernels are queued on the context's
 * stream, where every later call on this context is ordered after them. For pageable `img` (any ordinary host buffer) the call
 * returns once the image has left the caller's buffer; a page-locked `img` must stay unmodified until the next synchronising call
 * (dsdtm_sync or any call that returns results). Errors of the queued work surface at that call. */
int dsdtm_frame_upload_pyramid_async(dsdtm_ctx* ctx, int slot, const uint8_t* img, int stride);
/* batched: n dense (stride == width) images into slots first_slot .. first_slot+n-1; n <= DSDTM_MAX_BATCH_FRAMES */
int dsdtm_frames_upload_pyramid(dsdtm_ctx* ctx, int first_slot, int n, const uint8_t* imgs);
/* device-resident variant: level 0 of the n slots is already in HBM (e.g. written by a previous upload); rebuild levels.
 * n <= DSDTM_MAX_BATCH_FRAMES */
int dsdtm_frames_build_pyramid(dsdtm_ctx* ctx, int first_slot, int n);
/* parity helper: copy one level of a slot back (dense w*h bytes) */
/* Raw upload of ONE level image (w_level x h_level) into a slot, no pyramid: for callers that hold an image that is not a level-0
 * frame, e.g. the static Feature_Alignment::Align2DGaussNewton(const cv::Mat&, ...) (ref: include/Feature_alignment.h:85), which may
 * be handed any level of any pyramid. The other levels of the slot are left as they are. */
int dsdtm_frame_upload_level(dsdtm_ctx* ctx, int slot, int level, const uint8_t* img, int stride);
int dsdtm_frame_download_level(dsdtm_ctx* ctx, int slot, int level, uint8_t* out);

/* ---------------------------------------------------------------- (b) FAST + grid cells -------------------- */
/* replaces the per-level loop of Feature_detector::detect (ref: src/Feature_detection.cpp:74-109): FAST-10 at
 * `barrier` (reference literal: 20) on every level, 3x3 non-max on the FAST score, Shi-Tomasi score, per-cell best
 * (strictly greater than seed_score; earliest level, then raster order, wins ties). occupied (grid_rows*grid_cols
 * bytes, may be NULL) = mvGrid_occupy. cells_out[grid_rows*grid_cols] in cell order; empty cells = {0,0,0,seed_score}.
 * The sort and mask-circle selection that follow (ref: :111-150) are dsdtm_detect / dsdtm_detect_batch below. */
int dsdtm_fast_cells(dsdtm_ctx* ctx, int slot, int barrier, float seed_score, const uint8_t* occupied,
                     dsdtm_corner* cells_out);
/* batched over n consecutive slots (n <= max_batch and <= DSDTM_MAX_BATCH_FRAMES); occupied (may be NULL) and cells_out are
 * n * grid_rows*grid_cols */
int dsdtm_fast_cells_batch(dsdtm_ctx* ctx, int first_slot, int n, int barrier, float seed_score,
                           const uint8_t* occupied, dsdtm_corner* cells_out);
/* parity helper replacing fast_corner_detect_10[_sse2] + fast_corner_score_10 + fast_nonmax_3x3
 * (ref: Thirdparty/fast/include/fast/fast.h:20-29): dense maps for one level, w*h bytes each.
 * score[i] = FAST score (>= barrier) if pixel i is a corner else 0; nonmax[i] = 1 if it survives 3x3 non-max. */
int dsdtm_fast_score_map(dsdtm_ctx* ctx, int slot, int level, int barrier, uint8_t* score, uint8_t* nonmax);
int dsdtm_grid_dims(const dsdtm_ctx* ctx, int* rows, int* cols);

/* cv::circle(mask, px, radius, 0, -1): a filled circle painted into a detection mask before the selection. The centre is rounded
 * with cvRound on the device, so callers pass Feature::mpx as it is. 0 <= radius <= 64. */
typedef struct {
    float   px[2];
    int32_t radius;
    int32_t reserved;
} dsdtm_circle; /* 16 bytes */

/* replaces all of Feature_detector::detect (ref: src/Feature_detection.cpp:69-154) for the n consecutive slots first_slot..: FAST
 * with the reference's literal barrier 20 and the per-cell best above detection_threshold (as dsdtm_fast_cells), then the score sort
 * and the mask-circle selection on the device (detect_select_kernel), then one copy back. Per frame i:
 *   occupied   (n * grid_rows*grid_cols bytes, may be NULL) = mvGrid_occupy;
 *   masks      (n * height*width bytes, may be NULL = all 255) = mImgMask after Frame::Set_Mask; a pixel is free iff it is 255;
 *   circles    (n * circle_stride records, may be NULL) with n_circles[i] <= circle_stride: painted into the mask first;
 *   max_new[i] = Max_fts - mvFeatures.size(); a value <= 0 selects nothing (the early return of detect);
 *   out        (n * out_stride corners) receives n_out[i] corners in Add_Feature order; max_new[i] <= out_stride;
 *   exact_path (n bytes, may be NULL) = 1 where two cells above 20 tied and the frame was ordered by the restatement of libstdc++'s
 *              std::sort the reference's selection depends on, 0 where the parallel ranking was exact.
 * The result equals the reference's std::sort + walk bit for bit, including the order of tied scores. The device mask buffer is
 * allocated by the first call that passes masks. DSDTM_E_ARG (nothing launched) for a slot out of range, n > max_batch or
 * DSDTM_MAX_BATCH_FRAMES,
 * max_new > out_stride, a radius out of range, NULL out / n_out / max_new, or a frame geometry beyond 752 x 480 pixels. The
 * device time is counted under DSDTM_STAGE_FAST. */
int dsdtm_detect_batch(dsdtm_ctx* ctx, int first_slot, int n, float detection_threshold, const uint8_t* occupied, const uint8_t* masks,
                       const dsdtm_circle* circles, int circle_stride, const int* n_circles, const int* max_new, int out_stride,
                       dsdtm_corner* out, int* n_out, uint8_t* exact_path);
/* the same for one slot; inputs travel in one host-to-device copy and outputs in one copy back. circles / mask / occupied may be
 * NULL. Returns the selected corner count in *n_out. */
int dsdtm_detect(dsdtm_ctx* ctx, int slot, float detection_threshold, const uint8_t* occupied, const uint8_t* mask,
                 const dsdtm_circle* circles, int n_circles, int max_new, dsdtm_corner* out, int* n_out, uint8_t* exact_path);

/* ---------------------------------------------------------------- (c) sparse image alignment --------------- */
/* replaces Sprase_ImgAlign::Run's level loop: GetJocabianMat + GaussNewtonSolver for levels max_level-1 .. min_level
 * (ref: src/Sprase_ImageAlign.cpp:43-55,62-166,240-344). pose_c2r_in = T_cur * T_ref^-1 (ref: :43); the caller composes
 * pose_c2r_out * T_ref (ref: :57). *n_tracked = Run's return value. log (may be NULL) receives one entry per iteration. */
int dsdtm_sparse_align(dsdtm_ctx* ctx, int ref_slot, int cur_slot, const dsdtm_ref_feat* feats, int n_feats,
                       const double ref_center[3], const double pose_c2r_in[7], int max_level, int min_level,
                       int max_iters, double pose_c2r_out[7], int* n_tracked, dsdtm_iter_log* log, int log_cap,
                       int* n_log);
/* batched over independent frame pairs (the sweep of BASELINE.json configs[4]). feats is n_pairs * feat_stride. */
int dsdtm_sparse_align_batch(dsdtm_ctx* ctx, int n_pairs, const int* ref_slots, const int* cur_slots,
                             const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats,
                             const double* ref_centers, const double* poses_in, int max_level, int min_level,
                             int max_iters, double* poses_out, int* n_tracked, dsdtm_iter_log* log,
                             int log_cap_per_pair, int* n_log);

/* ---------------------------------------------------------------- (d) feature alignment -------------------- */
/* replaces Feature_Alignment::Align2DGaussNewton for n patches against ONE current frame
 * (ref: src/Feature_alignment.cpp:318-417; include/Feature_alignment.h:85). level[i] = pyramid level searched,
 * patch10 = n x 100 bytes (mPatch_WithBoarder; the 8x8 mPatch is its interior, ref: :261-275),
 * px_io = n x 2 doubles in LEVEL coordinates (tCurPx), converged[i] = return value. */
int dsdtm_align2d_batch(dsdtm_ctx* ctx, int cur_slot, const int* level, const uint8_t* patch10, double* px_io, int n,
                        int max_iters, uint8_t* converged);
/* replaces Feature_Alignment::WarpAffine + GetPatchNoBoarder for n candidates (ref: src/Feature_alignment.cpp:206-275).
 * ref_slot[i] = frame slot of the reference keyframe, A = n x 4 doubles (row-major A_cur<-ref),
 * ref_px = n x 2 floats (Feature::mpx), ref_level / search_level per candidate, patch10_out = n x 100 bytes. */
int dsdtm_warp_affine_batch(dsdtm_ctx* ctx, const int* ref_slot, const double* A, const float* ref_px,
                            const int* ref_level, const int* search_level, int n, uint8_t* patch10_out);

/* ---------------------------------------------------------------- (f-1) fused candidate pipeline ---------- */
/* One candidate of Feature_Alignment::FindMatchDirect after the host-side observation lookup (MapPoint::Get_ClosetObs,
 * ref: src/MapPoint.cpp:133-174; src/Feature_alignment.cpp:135-140): everything SolveAffineMatrix reads. */
typedef struct {
    int    ref_slot;        /* frame slot of the reference keyframe's pyramid */
    int    ref_level;       /* reference Feature::mlevel */
    float  ref_px[2];       /* reference Feature::mpx */
    double ref_normal[3];   /* reference Feature::mNormal */
    double ref_point_w[3];  /* reference feature's Mpt->Get_Pose() (ref: :167) */
    double kf_center[3];    /* KeyFrame::Get_CameraCnt() */
    double pose_c2r[7];     /* T_cur * T_kf^-1 (ref: :181) */
    double px[2];           /* Candidate::mPx: reprojection of the map point into the current frame, level 0 */
} dsdtm_candidate;          /* 160 bytes */

/* replaces SolveAffineMatrix + GetBestSearchLevel + WarpAffine + GetPatchNoBoarder + Align2DGaussNewton of FindMatchDirect
 * (ref: src/Feature_alignment.cpp:142-156) for n candidates against ONE current frame, without returning to the host
 * between the stages. max_search_level = Camera.MaxPyraLevels - 3 (ref: :144). Outputs: px_out = n x 2 refined positions
 * scaled back to level 0 (ref: :154), level_out = search level (ref: :156), converged = return value; A_out (optional,
 * may be NULL) = n x 4 row-major affine matrices for inspection. */
int dsdtm_feature_align_batch(dsdtm_ctx* ctx, int cur_slot, const dsdtm_candidate* cands, int n, int max_search_level,
                              int max_iters, double* px_out, int* level_out, uint8_t* converged, double* A_out);

/* ---------------------------------------------------------------- (f-1) local map on the device ------------ */
/* The map walk that feeds FindMatchDirect -- Feature_Alignment::ReprojectPoint (ref: src/Feature_alignment.cpp:54-69) for
 * every local map point (Tracking::UpdateLocalMap, ref: src/Tracking.cpp:258-313) and MapPoint::Get_ClosetObs
 * (ref: src/MapPoint.cpp:133-174) with the IsInImage gate of :138 -- runs on flat snapshots of the local map, and chains
 * into the candidate pipeline above without returning to the host. The host snapshots the tables once per frame (the
 * mapper thread mutates the objects, SURVEY 8b "threading"). */
typedef struct {
    int32_t slot;           /* frame slot of the keyframe's pyramid */
    int32_t reserved;
    double  center[3];      /* KeyFrame::Get_CameraCnt() */
    double  pose_c2w[7];    /* KeyFrame::Get_Pose() */
} dsdtm_kf_view;            /* 88 bytes */
typedef struct {
    int32_t kf;             /* index into the dsdtm_kf_view table (key of MapPoint::mObservations) */
    int32_t level;          /* observing Feature::mlevel */
    float   px[2];          /* observing Feature::mpx */
    double  normal[3];      /* observing Feature::mNormal */
    double  point_w[3];     /* observing Feature::Mpt->Get_Pose() (ref: src/Feature_alignment.cpp:167) */
} dsdtm_obs;                /* 64 bytes */
typedef struct {
    double  point_w[3];     /* MapPoint::Get_Pose() */
    int32_t obs_begin;      /* first observation in the dsdtm_obs table ... */
    int32_t obs_count;      /* ... listed in the iteration order of MapPoint::mObservations (ties keep the first) */
} dsdtm_map_point;          /* 32 bytes */
enum { DSDTM_LM_IN_IMAGE = 1,   /* ReprojectPoint returned true (IsInImage(px, 8)) */
       DSDTM_LM_OBS_OK = 2,     /* Get_ClosetObs returned true (cos of the viewing angle >= 0.5) */
       DSDTM_LM_REF_OK = 4,     /* the observing feature passes IsInImage(px / 2^level, 5, level) (ref: :138) */
       DSDTM_LM_CONVERGED = 8 };/* Align2DGaussNewton returned true */
typedef struct {
    double  px_proj[2];     /* Frame::World2Pixel(point) = Candidate::mPx before alignment (level 0) */
    double  px[2];          /* after FindMatchDirect (ref: :154); == px_proj when the candidate was not aligned */
    int32_t cell;           /* grid cell of ReprojectPoint (:60-61), -1 when not in the image */
    int32_t obs;            /* chosen observation (index into the dsdtm_obs table), -1 when the point has none */
    int32_t flags;          /* DSDTM_LM_* */
    int32_t level;          /* search level (ref: :156), -1 when the candidate was not aligned */
} dsdtm_reproj;             /* 48 bytes */
/* pose_cur_c2w / cur_center: Frame::Get_Pose() / Frame::Get_CameraCnt() of the current frame. Every point with
 * IN_IMAGE|OBS_OK|REF_OK is aligned (SolveAffineMatrix .. Align2DGaussNewton, as dsdtm_feature_align_batch); the greedy,
 * mask-dependent selection of SearchLocalPoints (:71-121) stays with the caller. n_pts <= max_batch * max_patches. */
int dsdtm_local_map_align_batch(dsdtm_ctx* ctx, int cur_slot, const double pose_cur_c2w[7], const double cur_center[3],
                                const dsdtm_kf_view* kfs, int n_kfs, const dsdtm_obs* obs, int n_obs,
                                const dsdtm_map_point* pts, int n_pts, int max_search_level, int max_iters,
                                dsdtm_reproj* out);

/* ---------------------------------------------------------------- (f-3 / f-4) keyframe ingest ------------- */
/* Depth images live in their own small pool of raw 16-bit frames (option "depth_slots", default 4, allocated on first
 * use). The CV_32F image of Tracking::Track_RGBDCam (ref: src/Tracking.cpp:56, convertTo(CV_32F, 1/DepthScale)) is never
 * needed by the hot path: the <= 5 lookups per new feature convert on the fly with the same single rounding. */
int dsdtm_depth_upload(dsdtm_ctx* ctx, int depth_slot, const uint16_t* depth, int stride_bytes);
/* The float image itself for n consecutive depth slots (ref: src/Tracking.cpp:56); out = n*h*w floats on the host, or NULL
 * to leave the result in HBM (timing). */
int dsdtm_depth_convert_f32(dsdtm_ctx* ctx, int first_depth_slot, int n, float depth_scale, float* out);
enum { DSDTM_LIFT_SKIPPED = 0,   /* Feature::mbInitial was set: untouched (ref: src/Frame.cpp:140-141, src/Tracking.cpp:427-433) */
       DSDTM_LIFT_OK = 1,        /* undistorted, normal, depth and world point valid */
       DSDTM_LIFT_NO_DEPTH = 2 };/* undistorted + normal only: Get_FeatureDetph returned -1 (or no depth slot given) */
typedef struct {
    float   px[2];          /* Feature::mpx after Frame::UndistortFeatures (ref: src/Frame.cpp:94-150) */
    float   depth;          /* Frame::Get_FeatureDetph(px) (ref: src/Frame.cpp:200-224), -1 when none */
    int32_t status;         /* DSDTM_LIFT_* */
    double  normal[3];      /* Feature::mNormal = normalize(Pixel2Camera(px, 1)) (ref: src/Frame.cpp:146-147) */
    double  point_w[3];     /* Frame::UnProject(px, depth) (ref: src/Frame.cpp:152-157): the new MapPoint's position */
} dsdtm_lifted;             /* 64 bytes */
/* Tracking::CraeteKeyframe's per-feature arithmetic (ref: src/Tracking.cpp:412-464) for the n features of one frame in one
 * launch. dist = {k1,k2,p1,p2,k3} (ref: src/Camera.cpp:41-45); depth_slot < 0: undistort + normal only; initial may be NULL. */
int dsdtm_keyframe_lift(dsdtm_ctx* ctx, int depth_slot, const double pose_c2w[7], const float dist[5], float depth_scale,
                        const float* px_in, const uint8_t* initial, int n, dsdtm_lifted* out);

/* cv::createCLAHE(clip_limit, Size(tiles_x, tiles_y))->apply(img) -- the preprocessing the reference's drivers run in front
 * of the Frame constructor (ref: Test/test_Feature_detection.cpp:85-86, Test/test_Euroc.cpp:64, Test/test_Optimizer.cpp:75,
 * all with (3.0, 8x8)) -- fused with Frame::ComputeImagePyramid: the n dense raw images are equalised into level 0 of slots
 * first_slot.. and their pyramids are built. Bit-exact against OpenCV. The image size must be divisible by the tile grid
 * (OpenCV pads otherwise; not implemented), tiles_x <= 16, tile height >= 8, n <= DSDTM_MAX_BATCH_FRAMES. level0_out (optional,
 * may be NULL): the equalised images back on the host (n * h * w bytes). */
int dsdtm_frames_upload_clahe_pyramid(dsdtm_ctx* ctx, int first_slot, int n, const uint8_t* imgs, double clip_limit,
                                      int tiles_x, int tiles_y, uint8_t* level0_out);

/* ---------------------------------------------------------------- local-map selection (8f-1, the caller's half) ---- */
/* Tracking::GetCloseKeyFrames (ref: src/Tracking.cpp:315-345) and the ranking at the top of Tracking::UpdateLocalMap
 * (ref: :261-277). The reference walks EVERY key frame of the map and projects its map points into the current frame until one
 * is visible (Frame::isVisible, ref: src/Frame.cpp:300-311) -- a key frame with no visible point costs all its points -- every
 * frame, on the tracking thread. Here the map lives in a device-resident table that is updated incrementally (a new key frame
 * appends its rows; a bundle adjustment re-uploads the ranges it moved) and one launch answers for the whole map.
 * Point rows are KeyFrame::mvMapPoints in order; a null or exactly-zero map point is the row {0,0,0} (skipped as at :324-328). */
typedef struct {
    int32_t pt_begin, pt_count;   /* this key frame's rows of the point array */
    double  t[3];                 /* KeyFrame::Get_Pose().translation() (the rank key of :332 is the distance of the translations) */
} dsdtm_map_kf;                   /* 32 bytes */
/* (re)write key-frame rows [first_kf, first_kf + n_kfs) and point rows [first_point, first_point + n_points); the table grows */
int dsdtm_map_table_upload(dsdtm_ctx* ctx, int first_kf, int n_kfs, const dsdtm_map_kf* kfs, int first_point, int n_points,
                           const double* points_w);
/* over key-frame rows [0, n_kfs): visible[k] = the key frame has a map point visible in the current frame (it enters tClose_kfs),
 * dist[k] = its rank key (0 when not visible); local[0 .. *n_local) = the first max_local (10 in the reference) visible key frames
 * by ascending distance, ties in row order (std::list::sort is stable) = mvpLocalKeyFrames. visible / dist may be NULL. */
int dsdtm_close_keyframes(dsdtm_ctx* ctx, const double pose_cur_c2w[7], int n_kfs, int max_local, uint8_t* visible, double* dist,
                          int32_t* local, int32_t* n_local);

/* ---------------------------------------------------------------- pose refinement after matching (8f-2) ---- */
/* Optimizer::PoseOptimization(FramePtr, int) (ref: src/Optimizer.cpp:20-101; residual / Jacobian / parameterisation
 * ref: include/Optimizer.h:129-258): motion-only bundle adjustment of the current frame over its matched map points -- the
 * step Tracking runs right after SearchLocalPoints (ref: src/Tracking.cpp:236). The reference delegates to ceres::Solve
 * (trust-region Levenberg-Marquardt, DENSE_SCHUR, CauchyLoss(1.0), max_num_iterations = 100 -- its tIterations argument is
 * ignored; pass max_iters = 100 for the same behaviour); the device routine runs that algorithm: a CTA of eight warps per frame
 * for up to one frame per SM, one warp per frame for sweeps (option "pose_opt_solo_max" moves the switch). Floating point:
 * results agree with a sequential evaluation to rounding (DESIGN.md 3f); a frame's result does not depend on its neighbours
 * in the batch, and is bit-reproducible from run to run for a given kernel choice.
 * One record per residual block, i.e. per feature of the frame with Mpt != NULL, !Mpt->IsBad() and mbInitial, in
 * mvFeatures order (ref: src/Optimizer.cpp:46-68). */
typedef struct {
    double  normal[3];   /* Feature::mNormal (the observation is normal.xy / normal.z)   ref: include/Optimizer.h:164-165 */
    double  point_w[3];  /* Feature::Mpt->Get_Pose()                                     ref: src/Optimizer.cpp:58 */
    int32_t level;       /* Feature::mlevel: the residual is divided by 1 << level       ref: include/Optimizer.h:167 */
    int32_t reserved;
} dsdtm_ba_obs;          /* 56 bytes */
enum { DSDTM_BA_FUNCTION_TOL = 0, DSDTM_BA_PARAMETER_TOL = 1, DSDTM_BA_GRADIENT_TOL = 2, DSDTM_BA_NO_CONVERGENCE = 3,
       DSDTM_BA_FAILURE = 4, DSDTM_BA_MIN_RADIUS = 5, DSDTM_BA_NO_RESIDUALS = 6 };
typedef struct {
    int32_t iterations;    /* minimizer iterations after iteration 0 (ceres summary.iterations.size() - 1) */
    int32_t termination;   /* DSDTM_BA_* : which of Ceres' stopping rules ended the solve */
    int32_t n_successful;  /* accepted steps */
    int32_t n_obs;
    double  initial_cost, final_cost;   /* sum over blocks of rho(|r|^2) / 2 */
} dsdtm_ba_summary;        /* 32 bytes */
/* n_frames independent frames: frame i owns obs[i * obs_stride .. + n_obs[i]), poses 7 doubles per frame (Frame::Get_Pose()
 * in, the argument of Frame::Set_Pose() out). res_norm (optional, n_frames * obs_stride): GetReprojectReidual() of the
 * final problem (ref: src/Optimizer.cpp:298-318), which the caller compares with LocalBAthreshhold / Camera.f to call
 * MapPoint::EraseFound (ref: :81-94). summaries optional. n_obs[i] <= DSDTM_BA_MAX_OBS. */
#define DSDTM_BA_MAX_OBS 4096
int dsdtm_pose_optimize_batch(dsdtm_ctx* ctx, int n_frames, const dsdtm_ba_obs* obs, int obs_stride, const int* n_obs,
                              const double* poses_in, int max_iters, double* poses_out, double* res_norm,
                              dsdtm_ba_summary* summaries);
/* one frame (the call PoseOptimization maps to) */
int dsdtm_pose_optimize(dsdtm_ctx* ctx, const dsdtm_ba_obs* obs, int n_obs, const double pose_in[7], int max_iters,
                        double pose_out[7], double* res_norm, dsdtm_ba_summary* summary);

/* ---------------------------------------------------------------- one call per tracked frame ---------------- */
/* Tracking::Track_RGBDCam's front end for one frame (ref: src/Tracking.cpp:57,199-224) as ONE call with ONE synchronisation:
 *   new Frame(img)                        -> upload + pyramid into cur_slot                     (ref: src/Frame.cpp:48-81)
 *   Sprase_ImgAlign::Run(cur, ref)        -> T_c2r from pose_c2r_in; cur pose = T_c2r * T_ref   (ref: src/Sprase_ImageAlign.cpp:29-60)
 *   UpdateLocalMap + SearchLocalPoints    -> ReprojectPoint / Get_ClosetObs / FindMatchDirect for every local map point with
 *                                            the NEW pose, which never leaves the device        (ref: src/Feature_alignment.cpp:54-158)
 * The greedy mask-dependent selection over the returned records stays with the caller, as for dsdtm_local_map_align_batch.
 * For maintainers who can change Tracking's call sequence; the three separate calls give identical results. */
typedef struct {
    int32_t ref_slot, cur_slot;
    const uint8_t* img; int32_t stride;              /* the new frame (host), bytes per row */
    const dsdtm_ref_feat* feats; int32_t n_feats;    /* features of the reference frame (as for dsdtm_sparse_align) */
    double ref_center[3];                            /* reference Frame::Get_CameraCnt() */
    double pose_ref_c2w[7];                          /* reference Frame::Get_Pose() */
    double pose_c2r_in[7];                           /* cur.Get_Pose() * ref.Get_Pose().inverse() (ref: src/Sprase_ImageAlign.cpp:43) */
    int32_t max_level, min_level, max_iters;         /* Sprase_ImgAlign constructor arguments */
    const dsdtm_kf_view* kfs; int32_t n_kfs;         /* local map snapshot (as for dsdtm_local_map_align_batch) */
    const dsdtm_obs* obs; int32_t n_obs;
    const dsdtm_map_point* pts; int32_t n_pts;
    int32_t max_search_level, align_iters;
} dsdtm_track_in;
typedef struct {
    double  pose_c2r[7];    /* Sprase_ImgAlign::mT_c2r */
    double  pose_cur_c2w[7];/* cur.Set_Pose(mT_c2r * ref.Get_Pose()) */
    double  cur_center[3];  /* cur.Get_CameraCnt() */
    int32_t n_tracked;      /* return value of Run */
    int32_t reserved;
} dsdtm_track_out;          /* 144 bytes */
int dsdtm_track_frame(dsdtm_ctx* ctx, const dsdtm_track_in* in, dsdtm_track_out* out, dsdtm_reproj* reproj /* n_pts */);

/* ---------------------------------------------------------------- device-resident map store -------------------------------- */
/* Tracking::UpdateLocalMap + Feature_Alignment::SearchLocalPoints' arithmetic as ONE call on a map that LIVES on the device
 * (ref: src/Tracking.cpp:257-345, src/Feature_alignment.cpp:54-69,128-158, src/MapPoint.cpp:133-174). The per-frame host work of the
 * reference -- a loop over every map point of the ten local key frames, a mutex-guarded Get_Pose per point, a std::map copy per
 * candidate -- becomes table maintenance at key-frame rate: a key frame appends its row and its features' rows once
 * (dsdtm_store_append_keyframe), map points are appended / updated when they are created, moved by a bundle adjustment or flagged bad
 * (dsdtm_store_set_points / dsdtm_store_update_points), and every frame makes one call (dsdtm_store_track). The batched chain writes back
 * into the store itself with dsdtm_batch_commit_store (found counts, bad flags, key frames and their new points). */
typedef struct {
    int32_t slot;           /* frame slot of the key frame's pyramid (KeyFrame::mvImg_Pyr) */
    int32_t feat_begin;     /* first row of this key frame in the feature table (filled by the library on append) */
    int32_t feat_count;
    int32_t reserved;
    double  pose_c2w[7];    /* KeyFrame::Get_Pose() */
    double  center[3];      /* KeyFrame::Get_CameraCnt() */
} dsdtm_store_kf;           /* 96 bytes */
typedef struct {
    int32_t mp;             /* row of the feature's map point in the point table (KeyFrame::mvMapPoints[i]), -1 = none */
    int32_t level;          /* Feature::mlevel */
    float   px[2];          /* Feature::mpx */
    double  normal[3];      /* Feature::mNormal */
    int32_t is_obs;         /* != 0: (key frame, this feature) is in MapPoint::mObservations of `mp` */
    int32_t next_obs;       /* library: next older observation of the same map point (feature-table row), -1 = end */
} dsdtm_store_feat;         /* 48 bytes */
typedef struct {
    double  point_w[3];     /* MapPoint::Get_Pose() */
    int32_t bad;            /* MapPoint::IsBad() */
    int32_t last_obs;       /* library: newest observation (feature-table row), -1 = none */
} dsdtm_store_point;        /* 32 bytes */
typedef struct {
    int32_t mp;             /* map point (row of the point table) */
    int32_t order;          /* (rank of the local key frame << 16) | feature index: the order in which UpdateLocalMap calls ReprojectPoint */
    dsdtm_reproj r;         /* as dsdtm_local_map_align_batch: projection, cell, chosen observation (feature-table row), flags, level, refined px */
} dsdtm_store_cand;         /* 56 bytes */
/* points [first, first + n): append (first == current size) or rewrite. bad may be NULL (= 0). Appended points start without observations. */
int dsdtm_store_set_points(dsdtm_ctx* ctx, int first, int n, const double* point_w, const int32_t* bad);
/* scattered update of existing points: positions (NULL = keep) and bad flags (NULL = keep) */
int dsdtm_store_update_points(dsdtm_ctx* ctx, const int32_t* ids, int n, const double* point_w, const int32_t* bad);
/* appends one key frame with its features (row = number of key frames before the call, returned in *row); the observation chains of
 * the features' map points are extended on the device */
int dsdtm_store_append_keyframe(dsdtm_ctx* ctx, const dsdtm_store_kf* kf, const dsdtm_store_feat* feats, int n_feats, int32_t* row);
/* pose / slot of an existing key frame (bundle adjustment moved it; its pyramid was re-uploaded into another slot) */
int dsdtm_store_set_keyframe(dsdtm_ctx* ctx, int row, int slot, const double pose_c2w[7], const double center[3]);
int dsdtm_store_clear(dsdtm_ctx* ctx);
/* MapPoint::mnFound: the store keeps one count per point row; a point appended by any path (dsdtm_store_set_points,
 * dsdtm_batch_commit_store) starts at 1, as MapPoint's constructor does; a rewritten row keeps its count. Scattered setter, as
 * dsdtm_store_update_points: found[i] becomes the count of point ids[i]. */
int dsdtm_store_set_found(dsdtm_ctx* ctx, const int32_t* ids, int n, const int32_t* found);
/* rows of the key-frame, feature and point tables (any pointer may be NULL) */
int dsdtm_store_size(const dsdtm_ctx* ctx, int32_t* n_kfs, int32_t* n_feats, int32_t* n_points);
/* Reads ranges of the tables as the library holds them (any output pointer may be NULL; found follows the point range): key frames
 * [kf_first, +n_kfs), features [feat_first, +n_feats), points and their found counts [point_first, +n_points). DSDTM_E_ARG for a range
 * past a table's end. Library fields: a feature's is_obs is the row of the key frame that observes its point + 1 (0 = no observation;
 * dsdtm_store_append_keyframe turns the caller's flag into this), next_obs the next older observing feature row of the same point (-1 =
 * end), a point's last_obs its newest observing feature row (-1 = none): walking last_obs -> next_obs lists MapPoint::mObservations
 * newest first. */
int dsdtm_store_fetch(dsdtm_ctx* ctx, int kf_first, int n_kfs, dsdtm_store_kf* kfs, int feat_first, int n_feats, dsdtm_store_feat* feats,
                      int point_first, int n_points, dsdtm_store_point* points, int32_t* found);
/* One frame: GetCloseKeyFrames over all key frames (a point of the key frame visible in the current frame), the max_local nearest by
 * |t_cur - t_kf| (stable in row order), every map point of those key frames once (first key frame in rank order wins, bad points
 * skipped), ReprojectPoint, and for the points inside the image Get_ClosetObs + the IsInImage gate + SolveAffineMatrix +
 * GetBestSearchLevel + WarpAffine + Align2DGaussNewton. Returns the local key frames in rank order and ONE record per point that landed
 * in the image (unordered; `order` restores the reference's insertion order, the caller sorts its cells by found count and replays the
 * mask-dependent greedy selection of SearchLocalPoints). cap = capacity of `out`; *n_out may exceed it (then only cap records are
 * written and the call returns DSDTM_E_ARG). Observations are walked newest first; with strict '>' on the cosine, exact ties keep the
 * newest (the reference: std::map<KeyFrame*> address order -- not reproducible). */
int dsdtm_store_track(dsdtm_ctx* ctx, int cur_slot, const double pose_cur_c2w[7], const double cur_center[3], int max_local,
                      int max_search_level, int align_iters, int32_t* local_rows, int32_t* n_local, dsdtm_store_cand* out, int cap,
                      int32_t* n_out);

/* Sprase_ImgAlign::Run + Tracking::UpdateLocalMap (+ the arithmetic of SearchLocalPoints) of one frame as ONE submission with one
 * synchronisation (ref: src/Tracking.cpp:199-224,257-313): sparse alignment of cur against ref, cur.Set_Pose(T_c2r * ref pose) on the
 * device (ref: src/Sprase_ImageAlign.cpp:57), then dsdtm_store_track with that pose. The current frame's pyramid must already be in
 * cur_slot (Frame's constructor uploads it). out: as dsdtm_track_frame; local_rows / cands / n_out: as dsdtm_store_track. */
typedef struct {
    int32_t ref_slot, cur_slot;
    int32_t n_feats, reserved;
    const dsdtm_ref_feat* feats;
    double  ref_center[3];
    double  pose_ref_c2w[7];
    double  pose_c2r_in[7];
    int32_t max_level, min_level, max_iters;
    int32_t max_local, max_search_level, align_iters;
} dsdtm_track_store_in;
int dsdtm_track_frame_store(dsdtm_ctx* ctx, const dsdtm_track_store_in* in, dsdtm_track_out* out, int32_t* local_rows, int32_t* n_local,
                            dsdtm_store_cand* cands, int cap, int32_t* n_out);

/* ---------------------------------------------------------------- batched front end (sweep / bench) -------- */
/* One "step" over n_pairs independent frame pairs: [pyramid(cur)] -> sparse align -> Align2D of the pair's patches
 * against its cur frame. Inputs are staged once (H2D), run() only launches kernels on HBM-resident data (CUDA-graph
 * replayed), fetch() copies results back. patches: n_pairs * patches_per_pair entries, patch_level < 0 = unused.
 * flags bit0: rebuild the cur pyramids from their level 0 inside run(); bit1: the refinement chain (dsdtm_batch_stage_map);
 * bit2 (with bit1): selection + pose optimization behind it (dsdtm_batch_stage_track); bit3 (with bit2): the key frame behind the
 * tracked pose (dsdtm_batch_stage_keyframe). n_pairs <= max_batch and <= DSDTM_MAX_BATCH_FRAMES (DSDTM_E_ARG, nothing staged). */
int dsdtm_batch_stage(dsdtm_ctx* ctx, int n_pairs, const int* ref_slots, const int* cur_slots,
                      const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats, const double* ref_centers,
                      const double* poses_in, int max_level, int min_level, int max_iters,
                      const uint8_t* patches10, const double* patch_px, const int* patch_level,
                      int patches_per_pair, int align_iters);
int dsdtm_batch_run(dsdtm_ctx* ctx, int flags);
/* The refinement chain of the reference as a batched stage (ref: src/Tracking.cpp:219-224,257-313 TrackWithLocalMap right after
 * Sprase_ImgAlign::Run; src/Feature_alignment.cpp:54-69,128-158): every pair's local map is its reference frame seen as one key
 * frame, whose features with map points (the staged dsdtm_ref_feat records, indices < points_per_pair) are the candidates. After
 * dsdtm_batch_stage, stage_map uploads the reference poses (n_pairs x 7, Frame::Get_Pose of the reference frames); then
 * dsdtm_batch_run(flags | 2) runs pyramid -> sparse alignment -> pose composition + reprojection + closest observation + gates ->
 * SolveAffineMatrix / GetBestSearchLevel -> WarpAffine -> Align2DGaussNewton for every candidate, all on the device, and
 * fetch_map returns n_pairs x points_per_pair records (obs = feature index; cell, flags, level, refined px as in
 * dsdtm_local_map_align_batch). The greedy per-cell selection of SearchLocalPoints stays with the caller unless flags bit 2 runs it
 * on the device (dsdtm_batch_stage_track below). */
int dsdtm_batch_stage_map(dsdtm_ctx* ctx, const double* poses_ref_c2w, int points_per_pair, int max_search_level, int align_iters);
int dsdtm_batch_fetch_map(dsdtm_ctx* ctx, dsdtm_reproj* reproj_out /* n_pairs x points_per_pair */);
/* The rest of Tracking::TrackWithLocalMap behind the chain (ref: src/Tracking.cpp:219-236): SearchLocalPoints' selection
 * (ref: src/Feature_alignment.cpp:71-121) and Optimizer::PoseOptimization (ref: src/Optimizer.cpp:20-101) on the device, so that
 * dsdtm_batch_run(flags | 2 | 4) ends in the tracked pose of every pair. Selection over a pair's records: cells in index order;
 * a cell's candidates (feature index order = the ReprojectPoint order) stably sorted by found count, descending; a candidate is
 * skipped when the mask at cvRound((float)px_proj) is painted, when OBS_OK | REF_OK is incomplete, when level < 0 or when it did
 * not converge; the first other candidate is the cell's match (Feature(px as Point2f, level), ref: :100-113) and paints a filled
 * circle of radius Camera.CellSize at cvRound of that px; 200 matches (the reference's literal, :75) end the search. The mask
 * starts all free (a new Frame). Then one dsdtm_ba_obs per match in match order (normal = Frame::Add_Feature's bearing of the
 * float px, point_w = the staged feature's point, the match level) and PoseOptimization from cur.Get_Pose() after Run
 * (T_c2r * T_ref, ref: src/Sprase_ImageAlign.cpp:57), with the solver of dsdtm_pose_optimize_batch for the same n_pairs. */
typedef struct {
    int32_t point;          /* feature index of the pair's staged dsdtm_ref_feat records (its map point) */
    float   px[2];          /* Feature::mpx of the new feature: Point2f of the refined position, level 0 */
    int32_t level;          /* Feature::mlevel: the search level */
} dsdtm_match;              /* 16 bytes */
#define DSDTM_TRACK_MAX_MATCHES 200
/* after dsdtm_batch_stage_map: found = n_pairs x points_per_pair MapPoint::mnFound counts (NULL = all 1, the value a new map point
 * starts with), max_iters = PoseOptimization's iteration cap (100 in the reference). Allocates the buffers of the selection and
 * the solve, which the replayed step owns. Calling dsdtm_batch_stage or dsdtm_batch_stage_map again drops this staging. */
int dsdtm_batch_stage_track(dsdtm_ctx* ctx, const int32_t* found, int max_iters);
/* after dsdtm_batch_run(flags | 2 | 4): poses_c2w_out = n_pairs x 7, the argument of Frame::Set_Pose after PoseOptimization;
 * n_matches = n_pairs; matches = n_pairs x DSDTM_TRACK_MAX_MATCHES (mvFeatures order, the first n_matches[i] valid);
 * res_norm = n_pairs x DSDTM_TRACK_MAX_MATCHES, GetReprojectReidual() at the final pose per match (ref: src/Optimizer.cpp:298-318):
 * the caller compares it with LocalBAthreshhold / Camera.f to call MapPoint::EraseFound (ref: :81-94) and keeps the found counts
 * itself, or, in store mode, dsdtm_batch_commit_store applies them to the store on the device; summaries = n_pairs. Every pointer may
 * be NULL. */
int dsdtm_batch_fetch_track(dsdtm_ctx* ctx, double* poses_c2w_out, int32_t* n_matches, dsdtm_match* matches, double* res_norm,
                            dsdtm_ba_summary* summaries);
/* Tracking::CraeteKeyframe behind the tracked pose (ref: src/Tracking.cpp:412-464), so that dsdtm_batch_run(flags | 2 | 4 | 8) ends in the
 * key frame the tracker would create from every wanted pair's cur frame. Per pair, after PoseOptimization:
 *   occupancy : Set_ExistingFeatures of the matches (ref: src/Feature_detection.cpp:43-50): cell int(px.y / (float)CellSize) * grid_cols
 *               + int(px.x / (float)CellSize); a cell index outside the grid is skipped (the reference's operator[] is undefined there);
 *   mask      : filled circles at cvRound of every match's px, radius Camera.CellSize (SearchLocalPoints, ref: src/Feature_alignment.cpp:
 *               100-113) and radius min_dist = Camera.Min_dist (Frame::Set_Mask, ref: src/Frame.cpp:286-298); no dynamic mask;
 *   detect    : Feature_detector::detect on the pair's cur slot as dsdtm_detect_batch (literal barrier 20, cells above
 *               detection_threshold, the literal std::sort order of tied scores) with max_new = max_fts - n_matches (<= 0: nothing);
 *   lift      : per new corner Frame::UndistortFeatures with dist = {k1,k2,p1,p2,k3}, the bearing, Get_FeatureDetph on depth slot
 *               depth_slots[i] (-1: none, DSDTM_LIFT_NO_DEPTH; raw depth / depth_scale) and UnProject with the pose after
 *               PoseOptimization, as dsdtm_keyframe_lift; the matches are mbInitial (SetPose) and are not lifted.
 * The key frame's mvFeatures are the matches of dsdtm_batch_fetch_track followed by the new corners; a new MapPoint belongs to every
 * corner whose record is DSDTM_LIFT_OK. NeedKeyframe stays with the caller: want (n_pairs bytes, NULL = all) selects the pairs; FAST
 * runs on the wanted pairs only, the others get no corners and cost one early exit per CTA of the other three kernels. Requires dsdtm_batch_stage_track (DSDTM_E_STATE otherwise); DSDTM_E_ARG,
 * with nothing enqueued, for a depth slot >= option depth_slots or < -1, a depth slot before the depth pool exists (dsdtm_depth_upload),
 * max_fts outside 1..DSDTM_MAX_FEATS_LIMIT, min_dist or cell_size above 64, or a frame geometry dsdtm_detect_batch rejects. Calling
 * dsdtm_batch_stage, _stage_map or _stage_track again drops this staging. Device time: detection under DSDTM_STAGE_FAST, the lift
 * under DSDTM_STAGE_INGEST. */
int dsdtm_batch_stage_keyframe(dsdtm_ctx* ctx, const int32_t* depth_slots /* n_pairs or NULL */, const uint8_t* want /* n_pairs or NULL */,
                               float detection_threshold, int min_dist, int max_fts, const float dist[5], float depth_scale);
/* after dsdtm_batch_run(flags | 8): n_new = n_pairs corner counts; corners and lifted = n_pairs x max_fts (Add_Feature order, rows past
 * n_new[i] zero); exact_path = n_pairs flags as in dsdtm_detect_batch. Every pointer may be NULL. */
int dsdtm_batch_fetch_keyframe(dsdtm_ctx* ctx, int32_t* n_new, dsdtm_corner* corners, dsdtm_lifted* lifted, uint8_t* exact_path);
/* The store-backed local map of the batched chain: instead of dsdtm_batch_stage_map's one-key-frame stand-in, every frame of the batch
 * runs Tracking::UpdateLocalMap on the context's map store (dsdtm_store_*), as dsdtm_store_track does for one frame (ref:
 * src/Tracking.cpp:219-345). After dsdtm_batch_stage, stage either dsdtm_batch_stage_map or this; flags bits 1, 2 and 3 then run on
 * whichever is staged, and staging one drops the other (dsdtm_batch_stage drops both). Per frame i, with the prior pose T_c2r * T_ref
 * (the sparse alignment's result times poses_ref_c2w[i], ref: src/Sprase_ImageAlign.cpp:57), on the key-frame rows [kf_range[2i],
 * kf_range[2i+1]) (kf_range NULL: every row of the store at the time of the run):
 *   GetCloseKeyFrames and UpdateLocalMap's ranking: the max_local nearest, stable in row order;
 *   every map point of those key frames once, the first key frame in rank order that lists it winning, bad points skipped;
 *   ReprojectPoint, Get_ClosetObs over the point's whole observation chain, the IsInImage gate, SolveAffineMatrix, GetBestSearchLevel,
 *   WarpAffine and Align2DGaussNewton
 * -- each with the semantics dsdtm_store_track documents. Frame i's records fill rows [i * cands_per_frame, ..) IN `order` (UpdateLocalMap's
 * ReprojectPoint order). A frame with more candidates than cands_per_frame keeps its first cands_per_frame records, gets n_matches -1 and
 * its prior pose from dsdtm_batch_fetch_track, and no key frame (flags bit 3); the other frames are unaffected.
 * Behind the chain (flags | 4), dsdtm_batch_stage_track's `found` has one entry per store point row at its call, shared by all frames
 * (NULL = all 1; rows appended later count 1); a dsdtm_match's `point` is the store point row and its dsdtm_ba_obs point is that
 * row's point_w; the selection sorts a cell's records by found count, descending, then by `order`. dsdtm_batch_stage_keyframe works on
 * top unchanged. Any store change (dsdtm_store_set_points / _update_points / _append_keyframe / _set_keyframe / _clear) drops the
 * captured steps, so the next dsdtm_batch_run runs on the changed map; the run returns DSDTM_E_STATE when the store no longer holds the
 * staged ranges. DSDTM_E_ARG, with nothing enqueued, for a range outside the store, max_local outside 1..16, cands_per_frame outside
 * 1..max_patches, an empty store, or a range length and local map whose prelude does not fit one CTA's shared memory (9 bytes per key
 * frame of the longest range + 32 bytes per 3 features of max_local * the largest key frame, rounded up to a power of two; about 20 k
 * key frames of 300 features). LIMIT: a range longer than that is refused, not split over CTAs; with kf_range NULL a store that grows
 * past it makes the next dsdtm_batch_run return DSDTM_E_ARG. DSDTM_E_STATE without dsdtm_batch_stage. Device time: the prelude and the candidates under
 * DSDTM_STAGE_LOCAL_MAP. */
int dsdtm_batch_stage_store(dsdtm_ctx* ctx, const double* poses_ref_c2w /* n_pairs x 7 */, const int32_t* kf_range /* n_pairs x 2 or NULL */,
                            int max_local, int max_search_level, int align_iters, int cands_per_frame);
/* after dsdtm_batch_run(flags | 2) in store mode: local_rows = n_pairs x 16 (the local key frames' store rows in rank order, -1 past
 * n_local[i]); cands = n_pairs x cands_per_frame records in `order` (rows past min(n_cand[i], cands_per_frame) zero); n_cand = the true
 * candidate count, which may exceed cands_per_frame. Every pointer may be NULL. */
int dsdtm_batch_fetch_store(dsdtm_ctx* ctx, int32_t* local_rows, int32_t* n_local, dsdtm_store_cand* cands, int32_t* n_cand);
/* dsdtm_batch_stage_track in store mode with live found counts: the selection reads the store's own counts (dsdtm_store_set_found,
 * dsdtm_batch_commit_store) at every run instead of a host snapshot. DSDTM_E_STATE without dsdtm_batch_stage_store; otherwise as
 * dsdtm_batch_stage_track, which keeps its snapshot semantics (NULL = all 1). */
int dsdtm_batch_stage_track_live(dsdtm_ctx* ctx, int max_iters);
/* Commits what the frames of the last dsdtm_batch_run with flags 7 or 15 in store mode did to the map store, in frame order, on the device
 * (ref: src/Feature_alignment.cpp:106, src/Optimizer.cpp:81-94, src/Tracking.cpp:412-464):
 *   found : for every frame with n_matches >= 0, +1 for each match's point (IncreaseFound); then -1 for each match i with
 *           res_norm[i] > outlier_threshold (strict; pass LocalBAthreshhold / Camera.f, compared in double) unless its point was bad when
 *           the commit started (EraseFound); every matched point whose count ends <= 0 gets bad = 1. The bad flags and counts are read
 *           when the commit starts, not when the step ran, on purpose: the walk never lists a bad point, so for the tracker the two are
 *           the same, and a caller that changes the store between the run and the commit (dsdtm_store_set_found, a point flagged bad by
 *           LocalMapping) gets what the reference's EraseFound loop, running after that change, would do. Residual block i is match i: a new
 *           frame's features are exactly its matches and the walk never lists a bad point, so the block / feature index shift of the
 *           per-frame EraseFound loop (features without a point or with a bad one) cannot arise. A frame with n_matches -1 changes nothing.
 *   key frames (flags 15 only): every wanted frame with n_matches >= 0 becomes a key frame. Features in mvFeatures order: the matches
 *           (mp = the store point row, the match level and px, normal = the bearing PoseOptimization's observation used, observing), then
 *           the new corners (px and normal of the lifted record, the corner level; a DSDTM_LIFT_OK corner gets a new point at point_w,
 *           found 1, not bad, and observes it; a corner without depth has mp -1). Row: slot = the pair's cur slot (the store now names
 *           it: do not reuse it for a later cur frame while the key frame lives), pose_c2w = the pose after PoseOptimization, center =
 *           Get_CameraCnt() of that pose.
 *   rows  : features and new points are appended frame by frame in frame order; key frames are appended in frame order (kf_rows NULL) or
 *           fill the row kf_rows[i] that the caller reserved for wanted frame i as an EMPTY key frame (dsdtm_store_append_keyframe with no
 *           features: never close, never in a local map), e.g. inside the scene's own range of a tiled store. Entries of frames that are
 *           not wanted are ignored; a wanted frame that overflowed leaves its row empty.
 *   chains: the store equals, bit for bit, the one sequential calls build in frame order: dsdtm_store_set_points for the new points,
 *           dsdtm_store_append_keyframe per key frame (or the same rewrite of the reserved row), dsdtm_store_update_points for the bad
 *           flags; a point observed by several key frames of one commit is linked newest first above its older chain.
 * Per frame i: kf_row_out[i] = its key-frame row (-1 if none), point_first_out[i] = its first new point row (-1 without a key frame),
 * n_points_out[i] = its new points; any of them may be NULL. Frames of one step that share a map all read the counts the step started
 * with and their increments add up; the result equals the sequential tracker when each map has at most one frame per step (a later frame
 * of the same map would have seen the earlier frame's counts, bad flags and key frame). Cost: a point that k key frames of one commit
 * observe is linked by one thread in O(k log k) dependent loads (k = 1 in that layout, k = frames per map otherwise). A commit that writes a
 * key frame or reallocates a table drops the captured store-mode steps; one that writes none (every flags-7 commit, flags 15 with nothing
 * wanted) keeps them: its found counts and bad flags are read from device memory by the replay. It reserves the worst case before enqueuing (DSDTM_E_NOMEM: the store is unchanged) and synchronises once to read the new table sizes.
 * DSDTM_E_ARG, nothing enqueued, for a NaN threshold or, for a wanted frame, a reserved row outside the table, not empty or named twice.
 * DSDTM_E_STATE without a store-mode run with flags bit 2 since the last staging, after dsdtm_store_clear, or for a second commit. */
int dsdtm_batch_commit_store(dsdtm_ctx* ctx, float outlier_threshold, const int32_t* kf_rows /* n_pairs or NULL */, int32_t* kf_row_out,
                             int32_t* point_first_out, int32_t* n_points_out);
/* Sequences on the device: after a store-mode dsdtm_batch_run with flags 7 or 15 and its dsdtm_batch_commit_store, every frame that advances
 * becomes its own next reference frame, as Tracking::Track_RGBDCam's TrackWithLastFrame does (ref: src/Tracking.cpp:199-205: the reference
 * frame is the last frame, cur.Set_Pose(last.Get_Pose())). One kernel, one CTA per frame, rewrites the staged per-frame inputs the captured
 * step reads, so the next dsdtm_batch_run replays it on them:
 *   ref slot   = the frame's cur slot (its pyramid is built);          pose_ref = the pose after PoseOptimization;
 *   centre     = Get_CameraCnt() of that pose (the arithmetic the commit uses for a key frame's centre);
 *   prior      = identity (T_c2r of cur.Set_Pose(last.Get_Pose()));   cur slot = next_cur_slots[i];
 *   features   = the frame's mvFeatures as Sprase_ImgAlign::GetJocabianMat reads them next (ref: src/Sprase_ImageAlign.cpp:84-103): its matches
 *                in match order (px and level of the match, initial 1, normal = the bearing PoseOptimization used, point_w = the store's
 *                point_w of the match's point row -- a point the commit flagged bad stays: the reference tests the pointer, not IsBad); after
 *                flags 15 a frame that became a key frame continues with its new corners in Add_Feature order (px and normal of the lifted
 *                record, the corner level, initial = DSDTM_LIFT_OK, point_w = the lifted point or zero): the feature list the commit wrote.
 *                Rows past n_feats[i] are zero.
 * Held frames keep reference, pose, centre, prior and features; only their cur slot moves to next_cur_slots[i]: frames with n_matches -1
 * (candidate overflow) and frames with hold[i] != 0 (hold NULL = none). The Lost rule (< 20 tracked points after Run, ref: :208) and
 * NeedKeyframe stay with the caller, who reads n_tracked with dsdtm_batch_fetch and passes the decisions through hold and want_next.
 * want_next (NULL = unchanged) replaces dsdtm_batch_stage_keyframe's want mask for the next run; a change of the wanted count drops the
 * captured flags-8 steps (their FAST grid is sized by it), never the others. status_out[i] (NULL allowed) = DSDTM_ADV_*.
 * Writes only buffers the captured steps point at: nothing is dropped (except as above) and a steady flags-7 sequence is pure replays.
 * Every error returns before anything is enqueued, with the staged state unchanged. DSDTM_E_STATE: no store-mode flags 7/15 run, no commit
 * since it, a second advance, one-key-frame mode, want_next without dsdtm_batch_stage_keyframe. DSDTM_E_ARG: a next cur slot outside
 * max_frames, named twice, the slot of a key frame of the store (an empty reserved row names no slot: it is never close and never
 * local) or equal to a frame's reference slot after the advance; a staged
 * feat_stride below max(DSDTM_TRACK_MAX_MATCHES, max_fts) -- refused rather than truncated. Synchronises once. */
enum { DSDTM_ADV_ADVANCED = 0, DSDTM_ADV_KEYFRAME = 1, DSDTM_ADV_HELD_OVERFLOW = 2, DSDTM_ADV_HELD_CALLER = 3 };
int dsdtm_batch_advance(dsdtm_ctx* ctx, const int32_t* next_cur_slots /* n_pairs */, const uint8_t* hold /* n_pairs or NULL */,
                        const uint8_t* want_next /* n_pairs or NULL */, uint8_t* status_out /* n_pairs or NULL */);
/* Frame::Frame's image input for the staged step (ref: src/Frame.cpp:48-81) in one call: the n_pairs dense level-0 images (imgs, n_pairs x
 * height x width bytes) into the staged cur slots, and, when depth is not NULL, the n_pairs 16-bit depth images (dense, n_pairs x height x
 * width) into the frames' depth slots of dsdtm_batch_stage_keyframe (frames without one skip theirs). The pyramids are built by the run's
 * flags bit 0. cudaMemcpyAsync on the context's stream, one copy per frame or one for contiguous slots; pinned buffers are faster, pageable
 * ones work. Returns when the images are on the device. DSDTM_E_STATE without dsdtm_batch_stage (depth: without _stage_keyframe). */
int dsdtm_batch_upload_step(dsdtm_ctx* ctx, const uint8_t* imgs, const uint16_t* depth);
/* the staged per-frame inputs exactly as the next dsdtm_batch_run reads them (every pointer may be NULL): ref_slots / cur_slots / n_feats
 * n_pairs each, feats n_pairs x feat_stride, centers n_pairs x 3, poses_ref (the reference poses of store or map mode) and poses_in (the
 * sparse alignment's prior T_c2r) n_pairs x 7. DSDTM_E_STATE without dsdtm_batch_stage. */
int dsdtm_batch_fetch_ref(dsdtm_ctx* ctx, int32_t* ref_slots, int32_t* cur_slots, dsdtm_ref_feat* feats, int32_t* n_feats, double* centers,
                          double* poses_ref, double* poses_in);
int dsdtm_batch_fetch(dsdtm_ctx* ctx, double* poses_out, int* n_tracked, double* patch_px_out, uint8_t* patch_conv);
/* end-to-end step with HOST buffers: uploads the n_pairs cur images (dense, pinned recommended) into their cur slots,
 * stages the per-pair inputs, runs, and fetches -- copies overlapped with compute in chunks on internal streams. Both e2e entries
 * take n_pairs <= max_batch and <= DSDTM_MAX_BATCH_FRAMES (DSDTM_E_ARG before any copy). */
/* the same with the refinement chain of dsdtm_batch_stage_map instead of host patches: per pair only the current image, the
 * reference features and three small arrays go up, the poses / counts / per-candidate records come back */
int dsdtm_track_batch_e2e(dsdtm_ctx* ctx, int n_pairs, const uint8_t* cur_imgs, const int* ref_slots, const int* cur_slots,
                          const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats, const double* ref_centers,
                          const double* poses_ref_c2w, const double* poses_c2r_in, int max_level, int min_level, int max_iters,
                          int points_per_pair, int max_search_level, int align_iters, double* poses_c2r_out, int* n_tracked,
                          dsdtm_reproj* reproj_out);
int dsdtm_pair_batch_e2e(dsdtm_ctx* ctx, int n_pairs, const uint8_t* cur_imgs, const int* ref_slots,
                         const int* cur_slots, const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats,
                         const double* ref_centers, const double* poses_in, int max_level, int min_level,
                         int max_iters, const uint8_t* patches10, const double* patch_px, const int* patch_level,
                         int patches_per_pair, int align_iters, double* poses_out, int* n_tracked,
                         double* patch_px_out, uint8_t* patch_conv);
/* device time of the last dsdtm_batch_run / e2e call measured with CUDA events on the context's stream [ms] */
float dsdtm_last_run_ms(const dsdtm_ctx* ctx);
/* CUDA-event stopwatch on the context's stream (the stream every kernel of this context is launched on):
 * start records an event; stop records a second one, synchronises the stream and returns the elapsed ms (< 0 on error). */
int   dsdtm_timer_start(dsdtm_ctx* ctx);
float dsdtm_timer_stop(dsdtm_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* DSDTM_GPU_H */
