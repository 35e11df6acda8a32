// sequence_advance.cu -- dsdtm_batch_advance: after a committed store-mode step, every frame that advances becomes its own next reference
// frame, as Tracking::Track_RGBDCam's TrackWithLastFrame (ref: src/Tracking.cpp:199-205) does, on the device.
//
//   sequence_advance_kernel : one CTA per frame. Thread 0 moves the slots (ref = the old cur slot, cur = the next one), writes the pose after
//                             PoseOptimization as the reference pose, its Get_CameraCnt() (se3_inv_exact, the commit's key-frame centre) and
//                             the identity prior. All threads write the feature list Sprase_ImgAlign::GetJocabianMat reads next (ref:
//                             src/Sprase_ImageAlign.cpp:84-103): the matches, then, for a new key frame, its corners, then zero rows up to
//                             feat_stride. A held frame only gets its next cur slot. Which frames advance, as key frames or not, is decided on
//                             the host (dsdtm_batch_advance) and passed per frame in adv[n + f].
#include "ctx.cuh"
#include "se3_exact.cuh"

namespace dsdtm {

namespace {

static const int kAdvThreads = 256;

struct AdvArgs {
    int n, stride, kf_stride;
    const int* adv;                             // n next cur slots, then n DSDTM_ADV_* modes
    const int* nm; const dsdtm_match* match; const dsdtm_ba_obs* obs; const double* pose;
    const dsdtm_store_point* pts;
    const int* nnew; const dsdtm_corner* corners; const dsdtm_lifted* lifted;
    int* ref_slots; int* cur_slots; double* poses_ref; double* centers; double* poses_in;
    dsdtm_ref_feat* feats; int* n_feats;
};

__global__ void __launch_bounds__(kAdvThreads) sequence_advance_kernel(const AdvArgs a)
{
    const int f = blockIdx.x, t = threadIdx.x;
    const int mode = a.adv[a.n + f];
    if (mode == DSDTM_ADV_HELD_OVERFLOW || mode == DSDTM_ADV_HELD_CALLER) {
        if (t == 0) a.cur_slots[f] = a.adv[f];
        return;
    }
    const int nm = a.nm[f];
    const int n_new = mode == DSDTM_ADV_KEYFRAME ? a.nnew[f] : 0;
    const int nf = nm + n_new;
    if (t == 0) {
        const double* P = a.pose + 7 * (size_t)f;
        double inv[7];
        se3_inv_exact(P, inv);                                       // Frame::Get_CameraCnt()
        a.ref_slots[f] = a.cur_slots[f];
        a.cur_slots[f] = a.adv[f];
#pragma unroll
        for (int q = 0; q < 7; ++q) { a.poses_ref[7 * (size_t)f + q] = P[q]; a.poses_in[7 * (size_t)f + q] = q ? 0.0 : 1.0; }
#pragma unroll
        for (int q = 0; q < 3; ++q) a.centers[3 * (size_t)f + q] = inv[4 + q];
        a.n_feats[f] = nf;
    }
    dsdtm_ref_feat* R = a.feats + (size_t)f * a.stride;
    for (int j = t; j < a.stride; j += kAdvThreads) {
        dsdtm_ref_feat o;
        if (j < nm) {                                                // a match: Feature(px, level) with its map point, mbInitial
            const size_t i = (size_t)f * DSDTM_TRACK_MAX_MATCHES + j;
            const dsdtm_match m = a.match[i];
            o.px[0] = m.px[0]; o.px[1] = m.px[1]; o.level = m.level; o.initial = 1;
            const dsdtm_store_point& p = a.pts[m.point];
#pragma unroll
            for (int k = 0; k < 3; ++k) { o.normal[k] = a.obs[i].normal[k]; o.point_w[k] = p.point_w[k]; }
        } else if (j < nf) {                                         // a new corner of the key frame (Add_Feature order)
            const size_t i = (size_t)f * a.kf_stride + (j - nm);
            const dsdtm_lifted l = a.lifted[i];
            const bool ok = l.status == DSDTM_LIFT_OK;
            o.px[0] = l.px[0]; o.px[1] = l.px[1]; o.level = a.corners[i].level; o.initial = ok ? 1 : 0;
#pragma unroll
            for (int k = 0; k < 3; ++k) { o.normal[k] = l.normal[k]; o.point_w[k] = ok ? l.point_w[k] : 0.0; }
        } else {
            o.px[0] = o.px[1] = 0.f; o.level = 0; o.initial = 0;
#pragma unroll
            for (int k = 0; k < 3; ++k) { o.normal[k] = 0.0; o.point_w[k] = 0.0; }
        }
        R[j] = o;
    }
}

}  // namespace

cudaError_t launch_sequence_advance(dsdtm_ctx* c, const int* adv_d, bool keyframes, cudaStream_t s)
{
    const auto& b = c->batch;
    AdvArgs a;
    a.n = b.n_pairs; a.stride = b.feat_stride; a.kf_stride = keyframes ? b.kf_max_fts : 0;
    a.adv = adv_d;
    a.nm = c->trk_nobs_d; a.match = c->trk_match_d; a.obs = c->trk_obs_d; a.pose = c->trk_pose_out_d;
    a.pts = c->st_pts_d;
    a.nnew = c->kf_nnew_d; a.corners = c->kf_corner_d; a.lifted = c->kf_lifted_d;
    a.ref_slots = c->ref_slots_d; a.cur_slots = c->cur_slots_d; a.poses_ref = c->poses_ref_d; a.centers = c->centers_d; a.poses_in = c->poses_in_d;
    a.feats = c->feats_d; a.n_feats = c->n_feats_d;
    sequence_advance_kernel<<<a.n, kAdvThreads, 0, s>>>(a);
    c->launches += 1;
    return cudaGetLastError();
}

}  // namespace dsdtm
