// local_map.cu -- SURVEY 8f-1: the map walk in front of FindMatchDirect, on flat snapshots of the local map.
//
//   kf_pose_kernel   : one thread per keyframe, T_c2r = T_cur * T_kf^-1 (ref: src/Feature_alignment.cpp:181) with Sophus
//                      semantics (inverse = conjugate + rotated negated translation; product normalises the quaternion).
//   local_map_kernel : one thread per map point:
//                        Frame::World2Pixel + Camera::IsInImage(px, 8) + cell index   (ref: src/Feature_alignment.cpp:54-69)
//                        MapPoint::Get_ClosetObs                                       (ref: src/MapPoint.cpp:133-174)
//                        IsInImage(ref px / 2^level, 5, level)                         (ref: src/Feature_alignment.cpp:138)
//                      and writes the dsdtm_candidate that candidate_prep_kernel (align2d.cu) consumes, so the chain
//                      reproject -> observation -> affine -> warp -> Align2D never returns to the host.
// fp64 in the reference's operation order, non-contracted (__dmul_rn / __dadd_rn), so every value that reaches the integer
// decisions (cvRound, cell index, strict '>' on the cosine) is the one the CPU computes. A few thousand points per frame:
// latency-bound by construction (one short dependent chain per thread); the point of the stage is removing the host round
// trip between sparse alignment and Align2D, not bandwidth.
#include "ctx.cuh"
#include "cand_prep.cuh"
#include "se3_exact.cuh"

namespace dsdtm {

namespace {

struct LmArgs {
    const dsdtm_kf_view* kfs; int n_kfs;
    const dsdtm_obs* obs;
    const dsdtm_map_point* pts; int n_pts;
    double pose_cur[7]; double cur_center[3];
    const double* pose_dev;     // optional: {pose_c2w[7], centre[3]} produced on the device (dsdtm_track_frame); overrides the two above
    float fx, fy, cx, cy;
    int width, height, cell_size, grid_cols;
    double* kf_pose;            // n_kfs x 7
    dsdtm_candidate* cand;      // n_pts
    dsdtm_reproj* out;          // n_pts
};

__global__ void __launch_bounds__(64) kf_pose_kernel(const LmArgs a)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.n_kfs) return;
    double inv[7], T[7], pc[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) pc[j] = a.pose_dev ? a.pose_dev[j] : a.pose_cur[j];
    se3_inv_exact(a.kfs[k].pose_c2w, inv);
    se3_mul_exact(pc, inv, T);
    double* o = a.kf_pose + 7 * k;
#pragma unroll
    for (int j = 0; j < 7; ++j) o[j] = T[j];
}

// Camera::IsInImage (ref: src/Camera.cpp:187-193): cvRound(float) is round-half-even; integer division of the image size.
// cvRound = cvtss2si: NaN (a map point at the camera centre projects to 0/0) gives INT_MIN and fails the test, whereas
// __float2int_rn(NaN) is 0 -- hence the explicit guard (pinned against the compiled reference: test_is_in_image_and_nan).
__device__ __forceinline__ bool in_image(float x, float y, int boundary, int level, int width, int height)
{
    if (!(x == x) || !(y == y)) return false;
    const int rx = __float2int_rn(x), ry = __float2int_rn(y);
    return rx >= boundary && rx < width / (1 << level) - boundary && ry >= boundary && ry < height / (1 << level) - boundary;
}

__global__ void __launch_bounds__(128) local_map_kernel(const LmArgs a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n_pts) return;
    const dsdtm_map_point mp = a.pts[i];
    const double P0 = mp.point_w[0], P1 = mp.point_w[1], P2 = mp.point_w[2];
    // Frame::World2Pixel (ref: src/Frame.cpp:318-323): Camera2Pixel(T_c2w * P) = fx * X / Z + cx
    double pc[7], cc[3];
#pragma unroll
    for (int j = 0; j < 7; ++j) pc[j] = a.pose_dev ? a.pose_dev[j] : a.pose_cur[j];
#pragma unroll
    for (int j = 0; j < 3; ++j) cc[j] = a.pose_dev ? a.pose_dev[7 + j] : a.cur_center[j];
    double q0, q1, q2;
    qrot_exact(pc, P0, P1, P2, q0, q1, q2);
    q0 = __dadd_rn(q0, pc[4]); q1 = __dadd_rn(q1, pc[5]); q2 = __dadd_rn(q2, pc[6]);
    const double u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
    const double v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
    int flags = 0, cell = -1, best = -1;
    if (in_image(__double2float_rn(u), __double2float_rn(v), 8, 0, a.width, a.height)) {          // ref: :58
        flags |= DSDTM_LM_IN_IMAGE;
        cell = (int)__ddiv_rn(v, (double)a.cell_size) * a.grid_cols + (int)__ddiv_rn(u, (double)a.cell_size);   // ref: :60-61
    }
    // MapPoint::Get_ClosetObs: direction point -> current camera, then the observation with the largest cosine (strict >)
    double f0 = __dsub_rn(cc[0], P0), f1 = __dsub_rn(cc[1], P1), f2 = __dsub_rn(cc[2], P2);
    double n = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(f0, f0), __dmul_rn(f1, f1)), __dmul_rn(f2, f2)));
    f0 = __ddiv_rn(f0, n); f1 = __ddiv_rn(f1, n); f2 = __ddiv_rn(f2, n);
    double best_cos = 0.0;
    if (mp.obs_count > 0) best = mp.obs_begin;                                                        // min_it = begin()
    for (int j = 0; j < mp.obs_count; ++j) {
        const double* O = a.kfs[a.obs[mp.obs_begin + j].kf].center;
        double r0 = __dsub_rn(O[0], P0), r1 = __dsub_rn(O[1], P1), r2 = __dsub_rn(O[2], P2);
        const double rn = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(r0, r0), __dmul_rn(r1, r1)), __dmul_rn(r2, r2)));
        r0 = __ddiv_rn(r0, rn); r1 = __ddiv_rn(r1, rn); r2 = __ddiv_rn(r2, rn);
        const double c = __dadd_rn(__dadd_rn(__dmul_rn(r0, f0), __dmul_rn(r1, f1)), __dmul_rn(r2, f2));
        if (c > best_cos) { best_cos = c; best = mp.obs_begin + j; }
    }
    dsdtm_candidate cd;
    cd.ref_slot = -1; cd.ref_level = 0;
    cd.px[0] = u; cd.px[1] = v;
    if (best >= 0) {
        if (!(best_cos < 0.5)) flags |= DSDTM_LM_OBS_OK;                                              // ref: MapPoint.cpp:170
        const dsdtm_obs ob = a.obs[best];
        const float sc = (float)(1 << ob.level);
        if (in_image(__fdiv_rn(ob.px[0], sc), __fdiv_rn(ob.px[1], sc), 5, ob.level, a.width, a.height)) flags |= DSDTM_LM_REF_OK;
        const int all = DSDTM_LM_IN_IMAGE | DSDTM_LM_OBS_OK | DSDTM_LM_REF_OK;
        if ((flags & all) == all) {
            const dsdtm_kf_view& kf = a.kfs[ob.kf];
            cd.ref_slot = kf.slot; cd.ref_level = ob.level;
            cd.ref_px[0] = ob.px[0]; cd.ref_px[1] = ob.px[1];
#pragma unroll
            for (int k = 0; k < 3; ++k) { cd.ref_normal[k] = ob.normal[k]; cd.ref_point_w[k] = ob.point_w[k]; cd.kf_center[k] = kf.center[k]; }
#pragma unroll
            for (int k = 0; k < 7; ++k) cd.pose_c2r[k] = a.kf_pose[7 * ob.kf + k];
        }
    }
    a.cand[i] = cd;
    dsdtm_reproj r;
    r.px_proj[0] = u; r.px_proj[1] = v; r.px[0] = u; r.px[1] = v;
    r.cell = cell; r.obs = best; r.flags = flags; r.level = -1;
    a.out[i] = r;
}

// Sprase_ImgAlign::Run's last line on the device (ref: src/Sprase_ImageAlign.cpp:57 cur.Set_Pose(T_c2r * ref.Get_Pose()); src/Frame.cpp:167-174
// Set_Pose: mOw = inverse().translation()): out = {pose_c2w[7], centre[3]} for the local-map kernels of the same call.
struct ComposeArgs { const double* t_c2r; double pose_ref[7]; double* out; };
__global__ void compose_pose_kernel(const ComposeArgs a)
{
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double T[7], Tc[7], inv[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) T[j] = a.t_c2r[j];
    se3_mul_exact(T, a.pose_ref, Tc);
    se3_inv_exact(Tc, inv);
#pragma unroll
    for (int j = 0; j < 7; ++j) a.out[j] = Tc[j];
    a.out[7] = inv[4]; a.out[8] = inv[5]; a.out[9] = inv[6];
}

// ---------------------------------------------------------------------------------------------------------------
// The refinement chain of a BATCH of independent frame pairs (bench / sweep: dsdtm_batch_run flags bit 1, dsdtm_track_batch_e2e):
// every pair's local map is its reference frame seen as ONE key frame, whose features with map points are the candidates --
// Tracking::TrackWithLocalMap right after a key frame (ref: src/Tracking.cpp:219-224,257-313). One thread per (pair, feature):
//   cur.Set_Pose(T_c2r * ref.Get_Pose())                       ref: src/Sprase_ImageAlign.cpp:57, src/Frame.cpp:167-174
//   ReprojectPoint: World2Pixel + IsInImage(px, 8) + cell      ref: src/Feature_alignment.cpp:54-69
//   Get_ClosetObs with the single observation (cos >= 0.5)     ref: src/MapPoint.cpp:133-174
//   IsInImage(ref px / 2^level, 5, level)                      ref: src/Feature_alignment.cpp:138
//   T_c2r' = cur.Get_Pose() * kf.Get_Pose().inverse()          ref: src/Feature_alignment.cpp:181
// and the dsdtm_candidate that candidate_prep_kernel consumes. Same non-contracted arithmetic as local_map_kernel / kf_pose_kernel /
// compose_pose_kernel (the pose composition is repeated per thread: ~150 flops, no extra launch, no extra pass over the poses).
struct PcArgs {
    const int* ref_slots; const dsdtm_ref_feat* feats; int feat_stride; const int* n_feats;
    const double* centers; const double* poses_ref; const double* poses_c2r;
    int pair0, n_pairs, ppp;
    float fx, fy, cx, cy;
    int width, height, cell_size, grid_cols;
    dsdtm_candidate* cand; dsdtm_reproj* out;
};

__global__ void __launch_bounds__(128) pair_candidates_kernel(const PcArgs a)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.n_pairs * a.ppp) return;
    const int pair = a.pair0 + t / a.ppp, j = t % a.ppp;
    const size_t i = (size_t)pair * a.ppp + j;
    dsdtm_candidate cd;
    cd.ref_slot = -1; cd.ref_level = 0; cd.px[0] = 0.0; cd.px[1] = 0.0;
    dsdtm_reproj r;
    r.px_proj[0] = r.px_proj[1] = r.px[0] = r.px[1] = 0.0; r.cell = -1; r.obs = -1; r.flags = 0; r.level = -1;
    const dsdtm_ref_feat ft = (j < a.n_feats[pair]) ? a.feats[(size_t)pair * a.feat_stride + j] : dsdtm_ref_feat{};
    if (j < a.n_feats[pair] && ft.initial) {                         // features without a map point are not in KeyFrame::GetMapPoints()
        double Tr[7], Tc2r[7], pc[7], inv[7], Tck[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) { Tr[k] = a.poses_ref[7 * pair + k]; Tc2r[k] = a.poses_c2r[7 * pair + k]; }
        se3_mul_exact(Tc2r, Tr, pc);                                 // cur pose (c2w)
        se3_inv_exact(pc, inv);                                      // cur centre = inverse().translation()
        const double cc0 = inv[4], cc1 = inv[5], cc2 = inv[6];
        se3_inv_exact(Tr, inv);
        se3_mul_exact(pc, inv, Tck);                                 // T_cur * T_kf^-1
        const double P0 = ft.point_w[0], P1 = ft.point_w[1], P2 = ft.point_w[2];
        double q0, q1, q2;
        qrot_exact(pc, P0, P1, P2, q0, q1, q2);
        q0 = __dadd_rn(q0, pc[4]); q1 = __dadd_rn(q1, pc[5]); q2 = __dadd_rn(q2, pc[6]);
        const double u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
        const double v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
        int flags = 0, cell = -1;
        if (in_image(__double2float_rn(u), __double2float_rn(v), 8, 0, a.width, a.height)) {
            flags |= DSDTM_LM_IN_IMAGE;
            cell = (int)__ddiv_rn(v, (double)a.cell_size) * a.grid_cols + (int)__ddiv_rn(u, (double)a.cell_size);
        }
        const double* O = a.centers + 3 * (size_t)pair;
        double f0 = __dsub_rn(cc0, P0), f1 = __dsub_rn(cc1, P1), f2 = __dsub_rn(cc2, P2);
        double n = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(f0, f0), __dmul_rn(f1, f1)), __dmul_rn(f2, f2)));
        f0 = __ddiv_rn(f0, n); f1 = __ddiv_rn(f1, n); f2 = __ddiv_rn(f2, n);
        double r0 = __dsub_rn(O[0], P0), r1 = __dsub_rn(O[1], P1), r2 = __dsub_rn(O[2], P2);
        const double rn = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(r0, r0), __dmul_rn(r1, r1)), __dmul_rn(r2, r2)));
        r0 = __ddiv_rn(r0, rn); r1 = __ddiv_rn(r1, rn); r2 = __ddiv_rn(r2, rn);
        const double cosv = __dadd_rn(__dadd_rn(__dmul_rn(r0, f0), __dmul_rn(r1, f1)), __dmul_rn(r2, f2));
        const double best_cos = (cosv > 0.0) ? cosv : 0.0;                                               // tMin_angle starts at 0, strict >
        if (!(best_cos < 0.5)) flags |= DSDTM_LM_OBS_OK;
        const float sc = (float)(1 << ft.level);
        if (in_image(__fdiv_rn(ft.px[0], sc), __fdiv_rn(ft.px[1], sc), 5, ft.level, a.width, a.height)) flags |= DSDTM_LM_REF_OK;
        cd.px[0] = u; cd.px[1] = v;
        const int all = DSDTM_LM_IN_IMAGE | DSDTM_LM_OBS_OK | DSDTM_LM_REF_OK;
        if ((flags & all) == all) {
            cd.ref_slot = a.ref_slots[pair]; cd.ref_level = ft.level;
            cd.ref_px[0] = ft.px[0]; cd.ref_px[1] = ft.px[1];
#pragma unroll
            for (int k = 0; k < 3; ++k) { cd.ref_normal[k] = ft.normal[k]; cd.ref_point_w[k] = ft.point_w[k]; cd.kf_center[k] = O[k]; }
#pragma unroll
            for (int k = 0; k < 7; ++k) cd.pose_c2r[k] = Tck[k];
        }
        r.px_proj[0] = u; r.px_proj[1] = v; r.px[0] = u; r.px[1] = v;
        r.cell = cell; r.obs = j; r.flags = flags;
    }
    a.cand[i] = cd;
    a.out[i] = r;
}

// After Align2D: fold (refined px * 2^level, level, converged) into the per-point records so that ONE copy returns everything.
__global__ void __launch_bounds__(128) local_map_finalize_kernel(dsdtm_reproj* __restrict__ out, const double* __restrict__ px,
                                                                 const int* __restrict__ level, const uint8_t* __restrict__ conv, int n, int i0)
{
    const int i = i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= i0 + n) return;
    const int L = level[i];
    if (L < 0) return;                                              // not aligned: px stays the projection, level -1
    const double sc = (double)(1 << L);                             // ref: :154 tPt = tCurPx * (1 << tBestLevel) (exact)
    out[i].px[0] = __dmul_rn(px[2 * i], sc); out[i].px[1] = __dmul_rn(px[2 * i + 1], sc);
    out[i].level = L;
    if (conv[i]) out[i].flags |= DSDTM_LM_CONVERGED;
}

}  // namespace

cudaError_t launch_local_map_finalize(dsdtm_ctx* c, int n_pts, cudaStream_t s, dsdtm_reproj* out_d, int i0)
{
    local_map_finalize_kernel<<<(n_pts + 127) / 128, 128, 0, s>>>(out_d ? out_d : c->lm_reproj_d, c->patch_px_d, c->patch_level_d, c->patch_conv_d, n_pts, i0);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_pair_candidates(dsdtm_ctx* c, int pair0, int n_pairs, int feat_stride, int ppp, cudaStream_t s)
{
    PcArgs a;
    a.ref_slots = c->ref_slots_d; a.feats = c->feats_d; a.feat_stride = feat_stride; a.n_feats = c->n_feats_d;
    a.centers = c->centers_d; a.poses_ref = c->poses_ref_d; a.poses_c2r = c->poses_out_d;
    a.pair0 = pair0; a.n_pairs = n_pairs; a.ppp = ppp;
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    a.width = c->cam.width; a.height = c->cam.height; a.cell_size = c->prm.cell_size; a.grid_cols = c->grid_cols;
    a.cand = c->cand_d; a.out = c->pair_reproj_d;
    const long long n = (long long)n_pairs * ppp;
    pair_candidates_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_compose_pose(dsdtm_ctx* c, const double* t_c2r_d, const double pose_ref_c2w[7], double* out10_d, cudaStream_t s)
{
    ComposeArgs a;
    a.t_c2r = t_c2r_d; a.out = out10_d;
    for (int k = 0; k < 7; ++k) a.pose_ref[k] = pose_ref_c2w[k];
    compose_pose_kernel<<<1, 32, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_local_map(dsdtm_ctx* c, const double pose_cur[7], const double cur_center[3], int n_kfs, int n_pts, cudaStream_t s,
                             const double* pose_dev)
{
    LmArgs a;
    a.pose_dev = pose_dev;
    a.kfs = c->lm_kfs_d; a.n_kfs = n_kfs; a.obs = c->lm_obs_d; a.pts = c->lm_pts_d; a.n_pts = n_pts;
    for (int k = 0; k < 7; ++k) a.pose_cur[k] = pose_cur ? pose_cur[k] : 0.0;
    for (int k = 0; k < 3; ++k) a.cur_center[k] = cur_center ? cur_center[k] : 0.0;
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    a.width = c->cam.width; a.height = c->cam.height; a.cell_size = c->prm.cell_size; a.grid_cols = c->grid_cols;
    a.kf_pose = c->lm_pose_d; a.cand = c->cand_d; a.out = c->lm_reproj_d;
    if (n_kfs > 0) kf_pose_kernel<<<(n_kfs + 63) / 64, 64, 0, s>>>(a);
    local_map_kernel<<<(n_pts + 127) / 128, 128, 0, s>>>(a);
    c->launches += 2;
    return cudaGetLastError();
}

// ---- Tracking::GetCloseKeyFrames on the device-resident map table (ref: src/Tracking.cpp:315-345, src/Frame.cpp:300-311).
// One warp per key frame: the lanes test 32 of its map points at a time (same non-contracted projection as above, boundary 0) and
// the warp stops at the first chunk with a visible point -- the reference's early break, 32 points wide. The work is one read of
// the point rows of the key frames that are NOT close (24 B per point) and one chunk of those that are.
namespace {
struct CkArgs {
    const dsdtm_map_kf* kfs; const double* pts; int n_kfs;
    double pose[7];
    float fx, fy, cx, cy; int width, height;
    uint8_t* visible; double* dist;
};

__global__ void __launch_bounds__(128) close_kf_kernel(const CkArgs a)
{
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= a.n_kfs) return;
    const int lane = threadIdx.x & 31;
    const dsdtm_map_kf kf = a.kfs[k];
    bool found = false;
    // software-pipelined: the next chunk's rows are requested before this chunk's vote, so the early-exit loop is not a chain of
    // dependent global loads (ncu: 9.9 long-scoreboard stalls per issued instruction without it)
    const double* rows = a.pts + 3 * (size_t)kf.pt_begin;
    double n0 = 0.0, n1 = 0.0, n2 = 0.0;
    if (lane < kf.pt_count) { n0 = rows[3 * lane]; n1 = rows[3 * lane + 1]; n2 = rows[3 * lane + 2]; }
    for (int base = 0; base < kf.pt_count && !found; base += 32) {
        const int i = base + lane;
        const double P0 = n0, P1 = n1, P2 = n2;
        const int j = i + 32;
        if (j < kf.pt_count) { n0 = rows[3 * (size_t)j]; n1 = rows[3 * (size_t)j + 1]; n2 = rows[3 * (size_t)j + 2]; }
        bool vis = false;
        if (i < kf.pt_count) {
            if (!(P0 == 0.0 && P1 == 0.0 && P2 == 0.0)) {                     // ref: :324-328
                double q0, q1, q2;
                qrot_exact(a.pose, P0, P1, P2, q0, q1, q2);
                q0 = __dadd_rn(q0, a.pose[4]); q1 = __dadd_rn(q1, a.pose[5]); q2 = __dadd_rn(q2, a.pose[6]);
                if (!(q2 < 0.0)) {                                              // ref: src/Frame.cpp:303
                    const double u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
                    const double v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
                    vis = in_image(__double2float_rn(u), __double2float_rn(v), 0, 0, a.width, a.height);
                }
            }
        }
        found = __any_sync(0xffffffffu, vis);
    }
    if (lane == 0) {
        a.visible[k] = found ? 1 : 0;
        const double d0 = __dsub_rn(a.pose[4], kf.t[0]), d1 = __dsub_rn(a.pose[5], kf.t[1]), d2 = __dsub_rn(a.pose[6], kf.t[2]);
        a.dist[k] = found ? sqrt(__dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2))) : 0.0;   // ref: :332
    }
}
}  // namespace

cudaError_t launch_close_keyframes(dsdtm_ctx* c, const double pose_cur[7], int n_kfs, cudaStream_t s)
{
    CkArgs a;
    a.kfs = c->mt_kfs_d; a.pts = c->mt_pts_d; a.n_kfs = n_kfs;
    for (int k = 0; k < 7; ++k) a.pose[k] = pose_cur[k];
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy; a.width = c->cam.width; a.height = c->cam.height;
    a.visible = c->mt_vis_d; a.dist = c->mt_dist_d;
    close_kf_kernel<<<(n_kfs + 3) / 4, 128, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------
// Device-resident map store (dsdtm_store_*): Tracking::UpdateLocalMap + the arithmetic of SearchLocalPoints without a per-frame host
// walk of the map. Tables: key frames (slot, pose, centre, feature range), features (map point, level, px, bearing, observation chain),
// map points (position, bad flag, newest observation).
namespace {

struct StArgs {
    const dsdtm_store_kf* kfs; dsdtm_store_feat* feats; dsdtm_store_point* pts; unsigned long long* claim;
    int n_kfs, max_local, cap, cur_slot, max_feats;
    unsigned epoch_inv;
    double pose[7], center[3];
    const double* pose_dev;                              // optional {pose_c2w[7], centre[3]} produced on the device (dsdtm_track_frame_store): overrides the two above
    float fx, fy, cx, cy;
    int width, height, cell_size, grid_cols;
    uint8_t* visible; double* dist; int* sel;            // sel[0] = n_local, sel[1..16] = local rows, sel[17] = n_cand
    dsdtm_candidate* cand; dsdtm_store_cand* out;
    int feat_begin, n_feats;                             // link kernel only
    const double* t_c2r_dev; double pose_ref[7]; double* pose10_out;   // prelude: compose the current pose from the sparse alignment's result
    CpArgs cp;                                           // candidate kernel: SolveAffineMatrix + GetBestSearchLevel for the record it has just built
    int max_search_level;
};

// observation chains: a new key frame's features are prepended to their map points' chains (one key frame observes a map point once)
__global__ void __launch_bounds__(128) store_link_kernel(const StArgs a)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.n_feats) return;
    dsdtm_store_feat& f = a.feats[a.feat_begin + j];
    f.next_obs = -1;
    if (f.mp >= 0 && f.is_obs) {
        f.next_obs = a.pts[f.mp].last_obs;
        a.pts[f.mp].last_obs = a.feat_begin + j;
    }
}

// Tracking::GetCloseKeyFrames (ref: src/Tracking.cpp:315-345): one warp per key frame, 32 of its map points per step, stop at the first
// visible one (Frame::isVisible: z >= 0 and IsInImage(px, 0)); distance = |t_cur - t_kf| of the POSE translations (ref: :332)
__global__ void __launch_bounds__(128) store_close_kf_kernel(const StArgs a)
{
    const int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= a.n_kfs) return;
    const int lane = threadIdx.x & 31;
    const dsdtm_store_kf& kf = a.kfs[k];
    double pose[7];
#pragma unroll
    for (int q = 0; q < 7; ++q) pose[q] = a.pose_dev ? a.pose_dev[q] : a.pose[q];
    bool found = false;
    for (int base = 0; base < kf.feat_count && !found; base += 32) {
        const int j = base + lane;
        bool vis = false;
        if (j < kf.feat_count) {
            const int mp = a.feats[kf.feat_begin + j].mp;
            if (mp >= 0) {
                const double P0 = a.pts[mp].point_w[0], P1 = a.pts[mp].point_w[1], P2 = a.pts[mp].point_w[2];
                if (!(P0 == 0.0 && P1 == 0.0 && P2 == 0.0)) {                  // ref: :324-328
                    double q0, q1, q2;
                    qrot_exact(pose, P0, P1, P2, q0, q1, q2);
                    q0 = __dadd_rn(q0, pose[4]); q1 = __dadd_rn(q1, pose[5]); q2 = __dadd_rn(q2, pose[6]);
                    if (!(q2 < 0.0)) {                                          // ref: src/Frame.cpp:303
                        const double u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
                        const double v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
                        vis = in_image(__double2float_rn(u), __double2float_rn(v), 0, 0, a.width, a.height);
                    }
                }
            }
        }
        found = __any_sync(0xffffffffu, vis);
    }
    if (lane == 0) {
        a.visible[k] = found ? 1 : 0;
        const double d0 = __dsub_rn(pose[4], kf.pose_c2w[4]), d1 = __dsub_rn(pose[5], kf.pose_c2w[5]), d2 = __dsub_rn(pose[6], kf.pose_c2w[6]);
        a.dist[k] = found ? sqrt(__dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2))) : 0.0;
    }
}

// UpdateLocalMap's ranking (ref: :266-277): the max_local smallest distances among the close key frames, ties in row order (the list is
// built in row order and std::list::sort is stable). One CTA: max_local rounds of a block-wide arg-min over (distance, row).
__global__ void __launch_bounds__(256) store_select_kernel(const StArgs a)
{
    __shared__ double s_d[256];
    __shared__ int s_i[256];
    __shared__ int s_taken[16];
    const int t = threadIdx.x;
    int n_sel = 0;
    for (int r = 0; r < a.max_local; ++r) {
        double bd = 0.0; int bi = -1;
        for (int k = t; k < a.n_kfs; k += 256) {
            if (!a.visible[k]) continue;
            bool taken = false;
            for (int q = 0; q < n_sel; ++q) taken |= (s_taken[q] == k);
            if (taken) continue;
            const double d = a.dist[k];
            if (bi < 0 || d < bd) { bd = d; bi = k; }                              // ascending k per thread: the first minimum is the lowest row
        }
        s_d[t] = bd; s_i[t] = bi;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (t < o) {
                const int j = s_i[t + o];
                if (j >= 0 && (s_i[t] < 0 || s_d[t + o] < s_d[t] || (s_d[t + o] == s_d[t] && j < s_i[t]))) { s_d[t] = s_d[t + o]; s_i[t] = j; }
            }
            __syncthreads();
        }
        const int win = s_i[0];
        __syncthreads();
        if (win < 0) break;
        if (t == 0) { s_taken[n_sel] = win; a.sel[1 + n_sel] = win; }
        ++n_sel;
        __syncthreads();
    }
    if (t == 0) { a.sel[0] = n_sel; a.sel[17] = 0; }
}

// every map point of the local key frames once: the FIRST (rank, feature) that lists it wins (ref: :283-297, mLastProjectedFrameId)
__global__ void __launch_bounds__(128) store_claim_kernel(const StArgs a)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (r >= a.sel[0]) return;
    const dsdtm_store_kf& kf = a.kfs[a.sel[1 + r]];
    if (j >= kf.feat_count) return;
    const int mp = a.feats[kf.feat_begin + j].mp;
    if (mp < 0 || a.pts[mp].bad) return;                                           // ref: :287-291
    atomicMin(a.claim + mp, ((unsigned long long)a.epoch_inv << 32) | (unsigned)((r << 16) | j));
}

// The three kernels above as ONE CTA of 1024 threads for maps of up to 1024 key frames (a launch per step costs more than the step):
// [compose the current pose from the sparse alignment's result, as compose_pose_kernel] -> close test, one warp per key frame ->
// ranking by counting (rank of k = number of visible (distance, row) pairs below its own: the stable ascending sort of ref: :266-277)
// -> claim. Results identical to store_close_kf_kernel + store_select_kernel + store_claim_kernel.
__global__ void __launch_bounds__(1024) store_prelude_kernel(const StArgs a)
{
    __shared__ double s_pose[10];
    __shared__ double s_dist[1024];
    __shared__ uint8_t s_vis[1024];
    __shared__ int s_sel[16];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) {
        if (a.t_c2r_dev) {
            double T[7], Tc[7], inv[7];
#pragma unroll
            for (int j = 0; j < 7; ++j) T[j] = a.t_c2r_dev[j];
            se3_mul_exact(T, a.pose_ref, Tc);
            se3_inv_exact(Tc, inv);
#pragma unroll
            for (int j = 0; j < 7; ++j) { s_pose[j] = Tc[j]; a.pose10_out[j] = Tc[j]; }
#pragma unroll
            for (int j = 0; j < 3; ++j) { s_pose[7 + j] = inv[4 + j]; a.pose10_out[7 + j] = inv[4 + j]; }
        } else {
#pragma unroll
            for (int j = 0; j < 7; ++j) s_pose[j] = a.pose_dev ? a.pose_dev[j] : a.pose[j];
        }
    }
    if (t < 16) s_sel[t] = -1;
    __syncthreads();
    double pose[7];
#pragma unroll
    for (int q = 0; q < 7; ++q) pose[q] = s_pose[q];
    for (int k = warp; k < a.n_kfs; k += 32) {
        const dsdtm_store_kf& kf = a.kfs[k];
        bool found = false;
        for (int base = 0; base < kf.feat_count && !found; base += 32) {
            const int j = base + lane;
            bool vis = false;
            if (j < kf.feat_count) {
                const int mp = a.feats[kf.feat_begin + j].mp;
                if (mp >= 0) {
                    const double P0 = a.pts[mp].point_w[0], P1 = a.pts[mp].point_w[1], P2 = a.pts[mp].point_w[2];
                    if (!(P0 == 0.0 && P1 == 0.0 && P2 == 0.0)) {
                        double q0, q1, q2;
                        qrot_exact(pose, P0, P1, P2, q0, q1, q2);
                        q0 = __dadd_rn(q0, pose[4]); q1 = __dadd_rn(q1, pose[5]); q2 = __dadd_rn(q2, pose[6]);
                        if (!(q2 < 0.0)) {
                            const double u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
                            const double v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
                            vis = in_image(__double2float_rn(u), __double2float_rn(v), 0, 0, a.width, a.height);
                        }
                    }
                }
            }
            found = __any_sync(0xffffffffu, vis);
        }
        if (lane == 0) {
            const double d0 = __dsub_rn(pose[4], kf.pose_c2w[4]), d1 = __dsub_rn(pose[5], kf.pose_c2w[5]), d2 = __dsub_rn(pose[6], kf.pose_c2w[6]);
            const double d = found ? sqrt(__dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2))) : 0.0;
            s_vis[k] = found ? 1 : 0; s_dist[k] = d;
            a.visible[k] = found ? 1 : 0; a.dist[k] = d;
        }
    }
    __syncthreads();
    const bool mine = t < a.n_kfs && s_vis[t];
    if (mine) {
        const double d = s_dist[t];
        int rank = 0;
        for (int j = 0; j < a.n_kfs; ++j)
            if (s_vis[j] && (s_dist[j] < d || (s_dist[j] == d && j < t))) ++rank;
        if (rank < a.max_local) { s_sel[rank] = t; a.sel[1 + rank] = t; }
    }
    const int n_sel = min(__syncthreads_count(mine), a.max_local);
    for (int r = 0; r < n_sel; ++r) {
        const dsdtm_store_kf& kf = a.kfs[s_sel[r]];
        for (int j = t; j < kf.feat_count; j += 1024) {
            const int mp = a.feats[kf.feat_begin + j].mp;
            if (mp < 0 || a.pts[mp].bad) continue;
            atomicMin(a.claim + mp, ((unsigned long long)a.epoch_inv << 32) | (unsigned)((r << 16) | j));
        }
    }
    if (t == 0) { a.sel[0] = n_sel; a.sel[17] = 0; }
}

// Frame::World2Pixel of a map point (ref: src/Frame.cpp:318-323), as every kernel of this file computes it
__device__ __forceinline__ void store_project(const StArgs& a, const double* pose, double P0, double P1, double P2, double& u, double& v)
{
    double q0, q1, q2;
    qrot_exact(pose, P0, P1, P2, q0, q1, q2);
    q0 = __dadd_rn(q0, pose[4]); q1 = __dadd_rn(q1, pose[5]); q2 = __dadd_rn(q2, pose[6]);
    u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
    v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
}

// A map point that landed in the image at (u, v) (ReprojectPoint returned true): its cell, Get_ClosetObs over its observation chain,
// the IsInImage gate, and the dsdtm_candidate record, handed to candidate_prep_one as entry i in the same thread
// (ref: src/Feature_alignment.cpp:54-69,128-141,160-204). Returns the record's reprojection fields.
__device__ __forceinline__ dsdtm_reproj store_candidate_one(const StArgs& a, int mp, const double* pose, const double* cc, double u, double v,
                                                            int i, int cur_slot)
{
    const double P0 = a.pts[mp].point_w[0], P1 = a.pts[mp].point_w[1], P2 = a.pts[mp].point_w[2];
    int flags = DSDTM_LM_IN_IMAGE;
    const int cell = (int)__ddiv_rn(v, (double)a.cell_size) * a.grid_cols + (int)__ddiv_rn(u, (double)a.cell_size);
    double f0 = __dsub_rn(cc[0], P0), f1 = __dsub_rn(cc[1], P1), f2 = __dsub_rn(cc[2], P2);
    double n = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(f0, f0), __dmul_rn(f1, f1)), __dmul_rn(f2, f2)));
    f0 = __ddiv_rn(f0, n); f1 = __ddiv_rn(f1, n); f2 = __ddiv_rn(f2, n);
    double best_cos = 0.0;
    int best = a.pts[mp].last_obs, best_kf = -1;
    for (int g = a.pts[mp].last_obs; g >= 0; g = a.feats[g].next_obs) {
        // the key frame of feature row g: rows are contiguous per key frame; the feature stores it in `is_obs - 1` (set on append)
        const int kr = a.feats[g].is_obs - 1;
        const double* O = a.kfs[kr].center;
        double r0 = __dsub_rn(O[0], P0), r1 = __dsub_rn(O[1], P1), r2 = __dsub_rn(O[2], P2);
        const double rn = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(r0, r0), __dmul_rn(r1, r1)), __dmul_rn(r2, r2)));
        r0 = __ddiv_rn(r0, rn); r1 = __ddiv_rn(r1, rn); r2 = __ddiv_rn(r2, rn);
        const double c = __dadd_rn(__dadd_rn(__dmul_rn(r0, f0), __dmul_rn(r1, f1)), __dmul_rn(r2, f2));
        if (c > best_cos) { best_cos = c; best = g; }
    }
    dsdtm_candidate cd;
    cd.ref_slot = -1; cd.ref_level = 0;
    cd.px[0] = u; cd.px[1] = v;
    if (best >= 0) {
        best_kf = a.feats[best].is_obs - 1;
        if (!(best_cos < 0.5)) flags |= DSDTM_LM_OBS_OK;
        const dsdtm_store_feat ob = a.feats[best];
        const float sc = (float)(1 << ob.level);
        if (in_image(__fdiv_rn(ob.px[0], sc), __fdiv_rn(ob.px[1], sc), 5, ob.level, a.width, a.height)) flags |= DSDTM_LM_REF_OK;
        const int all = DSDTM_LM_IN_IMAGE | DSDTM_LM_OBS_OK | DSDTM_LM_REF_OK;
        if ((flags & all) == all) {
            const dsdtm_store_kf& kf = a.kfs[best_kf];
            cd.ref_slot = kf.slot; cd.ref_level = ob.level;
            cd.ref_px[0] = ob.px[0]; cd.ref_px[1] = ob.px[1];
            // ref: :167 the reference feature's OWN map point (rf->Mpt->Get_Pose()): the observed point itself
            const int omp = ob.mp >= 0 ? ob.mp : mp;
#pragma unroll
            for (int k = 0; k < 3; ++k) { cd.ref_normal[k] = ob.normal[k]; cd.ref_point_w[k] = a.pts[omp].point_w[k]; cd.kf_center[k] = kf.center[k]; }
            double inv[7], T[7];
            se3_inv_exact(kf.pose_c2w, inv);
            se3_mul_exact(pose, inv, T);                                                             // ref: :181
#pragma unroll
            for (int k = 0; k < 7; ++k) cd.pose_c2r[k] = T[k];
        }
    }
    candidate_prep_one(a.cp, i, cd, cur_slot);
    dsdtm_reproj r;
    r.px_proj[0] = u; r.px_proj[1] = v; r.px[0] = u; r.px[1] = v;
    r.cell = cell; r.obs = best; r.flags = flags; r.level = -1;
    return r;
}

// ReprojectPoint for the claimed points; the ones inside the image become candidates (store_candidate_one)
__global__ void __launch_bounds__(128) store_candidates_kernel(const StArgs a)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (r >= a.sel[0]) return;
    const dsdtm_store_kf& kfr = a.kfs[a.sel[1 + r]];
    if (j >= kfr.feat_count) return;
    const int mp = a.feats[kfr.feat_begin + j].mp;
    if (mp < 0 || a.pts[mp].bad) return;
    const unsigned order = (unsigned)((r << 16) | j);
    if (a.claim[mp] != (((unsigned long long)a.epoch_inv << 32) | order)) return;
    double pose[7], cc[3];
#pragma unroll
    for (int q = 0; q < 7; ++q) pose[q] = a.pose_dev ? a.pose_dev[q] : a.pose[q];
#pragma unroll
    for (int q = 0; q < 3; ++q) cc[q] = a.pose_dev ? a.pose_dev[7 + q] : a.center[q];
    double u, v;
    store_project(a, pose, a.pts[mp].point_w[0], a.pts[mp].point_w[1], a.pts[mp].point_w[2], u, v);
    if (!in_image(__double2float_rn(u), __double2float_rn(v), 8, 0, a.width, a.height)) return;      // ref: :58
    const int slot_out = atomicAdd(a.sel + 17, 1);
    if (slot_out >= a.cap) return;
    dsdtm_store_cand o;
    o.mp = mp; o.order = (int)order;
    o.r = store_candidate_one(a, mp, pose, cc, u, v, slot_out, a.cur_slot);
    a.out[slot_out] = o;
}

// ---------------------------------------------------------------------------------------------------------------
// The batched chain on the map store (dsdtm_batch_stage_store): every frame of the batch runs UpdateLocalMap + SearchLocalPoints'
// arithmetic on the key-frame rows [begin, end) of the one store, with the prior pose T_c2r * T_ref of its sparse alignment.
//   store_batch_prelude_kernel    : one CTA per frame. Pose composition (as store_prelude_kernel), GetCloseKeyFrames over the range
//                                   (one warp per key frame), the counting rank (ties in row order), then the first-listing-wins walk:
//                                   every non-bad map point of the local key frames goes into a shared-memory open-addressing table
//                                   with the smallest order = (rank << 16) | feature index that lists it (atomicMin), and a second
//                                   pass in order emits the winners that ReprojectPoint puts in the image, compacted block-wide, so
//                                   record k of a frame is its k-th ReprojectPoint call. No global per-frame state, no epoch, no memset.
//   store_batch_candidates_kernel : grid (record blocks, frame): store_candidate_one for every emitted record; entries past the
//                                   frame's count are marked unused for warp_affine / Align2D.
// Shared memory of the prelude: 9 bytes per key frame of the longest range + 8 bytes per table slot, the table holding at least 4/3 of
// max_local * the largest feature count of a key frame (store_batch_smem).
static const int kSbThreads = 256, kSbWarps = kSbThreads / 32;

struct SbArgs {
    StArgs st;                                           // tables, camera, SolveAffineMatrix inputs (st.cp)
    const int2* range; int all_end, range_cap;           // per-frame [begin, end); null: [0, all_end)
    int n_pairs, max_local, cpf, tbits;
    const double* poses_c2r; const double* poses_ref;    // sparse alignment's T_c2r, reference Frame::Get_Pose
    const int* cur_slots;
    double* pose10; int* local; int* n_cand;
    dsdtm_store_cand* rec;
};

__global__ void __launch_bounds__(kSbThreads) store_batch_prelude_kernel(const SbArgs b)
{
    extern __shared__ __align__(16) unsigned char sb_smem[];
    __shared__ double s_pose[10];
    __shared__ int s_sel[16];
    __shared__ int s_wcnt[kSbWarps];
    const StArgs& a = b.st;
    const int f = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    int k0 = 0, k1 = b.all_end;
    if (b.range) { const int2 r = b.range[f]; k0 = r.x; k1 = r.y; }
    const int nk = k1 - k0, T = 1 << b.tbits;
    double* s_dist = reinterpret_cast<double*>(sb_smem);
    int* s_key = reinterpret_cast<int*>(s_dist + b.range_cap);
    unsigned* s_val = reinterpret_cast<unsigned*>(s_key + T);
    uint8_t* s_vis = reinterpret_cast<uint8_t*>(s_val + T);
    if (t == 0) {
        double T1[7], Tr[7], Tc[7], inv[7];
#pragma unroll
        for (int j = 0; j < 7; ++j) { T1[j] = b.poses_c2r[7 * (size_t)f + j]; Tr[j] = b.poses_ref[7 * (size_t)f + j]; }
        se3_mul_exact(T1, Tr, Tc);                                                 // ref: src/Sprase_ImageAlign.cpp:57
        se3_inv_exact(Tc, inv);
#pragma unroll
        for (int j = 0; j < 7; ++j) { s_pose[j] = Tc[j]; b.pose10[10 * (size_t)f + j] = Tc[j]; }
#pragma unroll
        for (int j = 0; j < 3; ++j) { s_pose[7 + j] = inv[4 + j]; b.pose10[10 * (size_t)f + 7 + j] = inv[4 + j]; }
    }
    if (t < 16) s_sel[t] = -1;
    for (int h = t; h < T; h += kSbThreads) { s_key[h] = -1; s_val[h] = 0xFFFFFFFFu; }
    __syncthreads();
    double pose[7];
#pragma unroll
    for (int q = 0; q < 7; ++q) pose[q] = s_pose[q];
    // GetCloseKeyFrames (ref: src/Tracking.cpp:315-345), as store_close_kf_kernel
    for (int q = warp; q < nk; q += kSbWarps) {
        const dsdtm_store_kf& kf = a.kfs[k0 + q];
        bool found = false;
        for (int base = 0; base < kf.feat_count && !found; base += 32) {
            const int j = base + lane;
            bool vis = false;
            if (j < kf.feat_count) {
                const int mp = a.feats[kf.feat_begin + j].mp;
                if (mp >= 0) {
                    const double P0 = a.pts[mp].point_w[0], P1 = a.pts[mp].point_w[1], P2 = a.pts[mp].point_w[2];
                    if (!(P0 == 0.0 && P1 == 0.0 && P2 == 0.0)) {
                        double q0, q1, q2;
                        qrot_exact(pose, P0, P1, P2, q0, q1, q2);
                        q0 = __dadd_rn(q0, pose[4]); q1 = __dadd_rn(q1, pose[5]); q2 = __dadd_rn(q2, pose[6]);
                        if (!(q2 < 0.0)) {
                            const double u = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fx, q0), q2), (double)a.cx);
                            const double v = __dadd_rn(__ddiv_rn(__dmul_rn((double)a.fy, q1), q2), (double)a.cy);
                            vis = in_image(__double2float_rn(u), __double2float_rn(v), 0, 0, a.width, a.height);
                        }
                    }
                }
            }
            found = __any_sync(0xffffffffu, vis);
        }
        if (lane == 0) {
            const double d0 = __dsub_rn(pose[4], kf.pose_c2w[4]), d1 = __dsub_rn(pose[5], kf.pose_c2w[5]), d2 = __dsub_rn(pose[6], kf.pose_c2w[6]);
            s_vis[q] = found ? 1 : 0;
            s_dist[q] = found ? sqrt(__dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2))) : 0.0;
        }
    }
    __syncthreads();
    // UpdateLocalMap's ranking (ref: :266-277): rank = visible (distance, row) pairs below this one's
    for (int q = t; q < nk; q += kSbThreads) {
        if (!s_vis[q]) continue;
        const double d = s_dist[q];
        int rank = 0;
        for (int j = 0; j < nk; ++j)
            if (s_vis[j] && (s_dist[j] < d || (s_dist[j] == d && j < q))) ++rank;
        if (rank < b.max_local) s_sel[rank] = k0 + q;
    }
    __syncthreads();
    int n_sel = 0;                                       // the ranks of the visible key frames are 0 .. n_visible - 1
    while (n_sel < b.max_local && s_sel[n_sel] >= 0) ++n_sel;
    if (t < 17) b.local[17 * (size_t)f + t] = t == 0 ? n_sel : (t - 1 < n_sel ? s_sel[t - 1] : -1);
    // every map point of the local key frames once: the smallest order that lists it (ref: :283-297, mLastProjectedFrameId)
    const unsigned hshift = 32u - (unsigned)b.tbits;
    for (int r = 0; r < n_sel; ++r) {
        const dsdtm_store_kf& kf = a.kfs[s_sel[r]];
        for (int j = t; j < kf.feat_count; j += kSbThreads) {
            const int mp = a.feats[kf.feat_begin + j].mp;
            if (mp < 0 || a.pts[mp].bad) continue;                                  // ref: :287-291
            unsigned h = ((unsigned)mp * 0x9E3779B1u) >> hshift;
            for (;;) {
                const int prev = atomicCAS(s_key + h, -1, mp);
                if (prev == -1 || prev == mp) { atomicMin(s_val + h, (unsigned)((r << 16) | j)); break; }
                h = (h + 1) & (unsigned)(T - 1);
            }
        }
    }
    __syncthreads();
    // the winners in order; ReprojectPoint (ref: :54-69) keeps those inside the image
    int base = 0;
    dsdtm_store_cand* R = b.rec + (size_t)f * b.cpf;
    for (int r = 0; r < n_sel; ++r) {
        const dsdtm_store_kf& kf = a.kfs[s_sel[r]];
        for (int j0 = 0; j0 < kf.feat_count; j0 += kSbThreads) {
            const int j = j0 + t;
            const unsigned order = (unsigned)((r << 16) | j);
            int mp = -1;
            bool win = false;
            if (j < kf.feat_count) {
                mp = a.feats[kf.feat_begin + j].mp;
                if (mp >= 0 && !a.pts[mp].bad) {
                    unsigned h = ((unsigned)mp * 0x9E3779B1u) >> hshift;
                    while (s_key[h] != mp) h = (h + 1) & (unsigned)(T - 1);
                    if (s_val[h] == order) {
                        double u, v;
                        store_project(a, pose, a.pts[mp].point_w[0], a.pts[mp].point_w[1], a.pts[mp].point_w[2], u, v);
                        win = in_image(__double2float_rn(u), __double2float_rn(v), 8, 0, a.width, a.height);
                    }
                }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, win);
            if (lane == 0) s_wcnt[warp] = __popc(bal);
            __syncthreads();
            int off = 0, tot = 0;
#pragma unroll
            for (int w = 0; w < kSbWarps; ++w) { const int c = s_wcnt[w]; off += w < warp ? c : 0; tot += c; }
            if (win) {
                const int pos = base + off + __popc(bal & ((1u << lane) - 1u));
                if (pos < b.cpf) { R[pos].mp = mp; R[pos].order = (int)order; }
            }
            base += tot;
            __syncthreads();
        }
    }
    if (t == 0) b.n_cand[f] = base;
}

__global__ void __launch_bounds__(128) store_batch_candidates_kernel(const SbArgs b)
{
    const int f = blockIdx.y, k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= b.cpf) return;
    const StArgs& a = b.st;
    const int n = min(b.n_cand[f], b.cpf);
    const int i = f * b.cpf + k;
    const int cur_slot = b.cur_slots[f];
    if (k >= n) {                                        // unused entry: warp_affine and Align2D skip it
        dsdtm_candidate cd;
        cd.ref_slot = -1; cd.ref_level = 0; cd.px[0] = 0.0; cd.px[1] = 0.0;
        candidate_prep_one(a.cp, i, cd, cur_slot);
        return;
    }
    double pose[7], cc[3];
#pragma unroll
    for (int q = 0; q < 7; ++q) pose[q] = b.pose10[10 * (size_t)f + q];
#pragma unroll
    for (int q = 0; q < 3; ++q) cc[q] = b.pose10[10 * (size_t)f + 7 + q];
    dsdtm_store_cand o = b.rec[i];
    double u, v;
    store_project(a, pose, a.pts[o.mp].point_w[0], a.pts[o.mp].point_w[1], a.pts[o.mp].point_w[2], u, v);
    o.r = store_candidate_one(a, o.mp, pose, cc, u, v, i, cur_slot);
    b.rec[i] = o;
}

// slots of the prelude's table for max_local key frames of the store's widest feature count
int store_batch_tbits(const dsdtm_ctx* c, int max_local)
{
    const long long n = (long long)max_local * std::max(c->st_max_feats, 1);
    int bits = 6;
    while ((1ll << bits) * 3 < n * 4) ++bits;
    return bits;
}

StArgs store_args(dsdtm_ctx* c)
{
    StArgs a;
    a.kfs = c->st_kfs_d; a.feats = c->st_feats_d; a.pts = c->st_pts_d; a.claim = c->st_claim_d;
    a.n_kfs = (int)c->st_kfs_n; a.max_local = 0; a.cap = 0; a.cur_slot = 0; a.max_feats = c->st_max_feats; a.epoch_inv = 0; a.pose_dev = nullptr;
    for (int k = 0; k < 7; ++k) a.pose[k] = 0.0;
    for (int k = 0; k < 3; ++k) a.center[k] = 0.0;
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    a.width = c->cam.width; a.height = c->cam.height; a.cell_size = c->prm.cell_size; a.grid_cols = c->grid_cols;
    a.visible = c->st_vis_d; a.dist = c->st_dist_d; a.sel = c->st_sel_d; a.cand = c->cand_d; a.out = c->st_out_d;
    a.feat_begin = 0; a.n_feats = 0;
    a.t_c2r_dev = nullptr; a.pose10_out = nullptr; a.max_search_level = 0;
    for (int k = 0; k < 7; ++k) a.pose_ref[k] = 0.0;
    a.cp.cand = nullptr; a.cp.n = 0; a.cp.cur_slot = 0; a.cp.max_search_level = 0; a.cp.i0 = 0; a.cp.cur_slots = nullptr; a.cp.ppp = 0;
    a.cp.fx = c->cam.fx; a.cp.fy = c->cam.fy; a.cp.cx = c->cam.cx; a.cp.cy = c->cam.cy;
    a.cp.A = c->wa_A_d; a.cp.ref_px = c->wa_px_d; a.cp.meta = c->wa_meta_d;
    a.cp.patch_level = c->patch_level_d; a.cp.patch_slot = c->patch_slot_d; a.cp.px_in = c->patch_px_in_d;
    return a;
}

}  // namespace

cudaError_t launch_store_link(dsdtm_ctx* c, int feat_begin, int n_feats, cudaStream_t s)
{
    if (n_feats <= 0) return cudaSuccess;
    StArgs a = store_args(c);
    a.feat_begin = feat_begin; a.n_feats = n_feats;
    store_link_kernel<<<(n_feats + 127) / 128, 128, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

// [pose composition ->] close key frames -> ranking -> claim, then candidates + SolveAffineMatrix / GetBestSearchLevel: two launches,
// nothing returns to the host. The caller chains warp_affine / Align2D over at most `cap` records with the device-side count
// (store_count_dev) and the store records as Align2D's extra output.
cudaError_t launch_store_track(dsdtm_ctx* c, const StoreTrackArgs& t, cudaStream_t s)
{
    StArgs a = store_args(c);
    a.n_kfs = t.n_kfs; a.max_local = t.max_local; a.cap = t.cap; a.cur_slot = t.cur_slot;
    a.epoch_inv = 0xFFFFFFFFu - c->st_epoch;
    for (int k = 0; k < 7; ++k) a.pose[k] = t.pose_cur[k];
    for (int k = 0; k < 3; ++k) a.center[k] = t.cur_center[k];
    a.pose_dev = t.pose_dev;
    a.t_c2r_dev = t.t_c2r_dev; a.pose10_out = t.pose10_out;
    for (int k = 0; k < 7; ++k) a.pose_ref[k] = t.pose_ref[k];
    a.cp.n = t.cap; a.cp.cur_slot = t.cur_slot; a.cp.max_search_level = t.max_search_level;
    const dim3 grid((unsigned)((std::max(c->st_max_feats, 1) + 127) / 128), (unsigned)t.max_local);
    if (t.n_kfs <= 1024) {
        store_prelude_kernel<<<1, 1024, 0, s>>>(a);
        c->launches += 1;
    } else {
        if (t.t_c2r_dev) {
            cudaError_t e = launch_compose_pose(c, t.t_c2r_dev, t.pose_ref, t.pose10_out, s);
            if (e != cudaSuccess) return e;
        }
        store_close_kf_kernel<<<(t.n_kfs + 3) / 4, 128, 0, s>>>(a);
        store_select_kernel<<<1, 256, 0, s>>>(a);
        store_claim_kernel<<<grid, 128, 0, s>>>(a);
        c->launches += 3;
    }
    if (t.t_c2r_dev) a.pose_dev = t.pose10_out;
    store_candidates_kernel<<<grid, 128, 0, s>>>(a);
    c->launches += 1;
    return cudaGetLastError();
}

const int* store_count_dev(dsdtm_ctx* c) { return c->st_sel_d + 17; }

size_t store_batch_smem(const dsdtm_ctx* c, int range_len, int max_local)
{
    const size_t cap = (size_t)((std::max(range_len, 1) + 1) & ~1);          // keeps the int table 8-byte aligned after the doubles
    return cap * sizeof(double) + ((size_t)8 << store_batch_tbits(c, max_local)) + cap;
}

cudaError_t store_batch_init(dsdtm_ctx* c)
{
    int max_smem = 0;
    cudaError_t e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(store_batch_prelude_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem - 1024);
    return e;
}

cudaError_t launch_store_batch(dsdtm_ctx* c, int n_pairs, bool all_rows, int range_len, int max_local, int cpf, int max_search_level, cudaStream_t s)
{
    SbArgs b;
    b.st = store_args(c);
    b.st.cp.n = n_pairs * cpf; b.st.cp.max_search_level = max_search_level;
    b.range = all_rows ? nullptr : c->sb_range_d; b.all_end = (int)c->st_kfs_n;
    b.range_cap = (std::max(range_len, 1) + 1) & ~1;
    b.n_pairs = n_pairs; b.max_local = max_local; b.cpf = cpf; b.tbits = store_batch_tbits(c, max_local);
    b.poses_c2r = c->poses_out_d; b.poses_ref = c->poses_ref_d; b.cur_slots = c->cur_slots_d;
    b.pose10 = c->sb_pose10_d; b.local = c->sb_local_d; b.n_cand = c->sb_ncand_d; b.rec = c->sb_rec_d;
    store_batch_prelude_kernel<<<n_pairs, kSbThreads, store_batch_smem(c, range_len, max_local), s>>>(b);
    store_batch_candidates_kernel<<<dim3((unsigned)((cpf + 127) / 128), (unsigned)n_pairs), 128, 0, s>>>(b);
    c->launches += 2;
    return cudaGetLastError();
}

}  // namespace dsdtm
