// store_commit.cu -- what the frames of one store-mode step did to the map (dsdtm_batch_commit_store): MapPoint::IncreaseFound on every
// match (ref: src/Feature_alignment.cpp:106), EraseFound on every outlier (ref: src/Optimizer.cpp:81-94) and, after flags 15, the key frames
// of Tracking::CraeteKeyframe (ref: src/Tracking.cpp:412-464) appended to the map store, all on the device.
//
//   commit_found_kernel : one CTA per frame. found[p] += 1 - (res_norm > threshold && !bad[p]) for every match of a tracked frame (n_matches
//                         >= 0); an integer sum, so the result does not depend on the order of the atomics. Counts the frame's feature rows
//                         (matches + new corners), new points (DSDTM_LIFT_OK corners) and key frame (wanted, tracked, flags 15).
//   commit_scan_kernel  : one CTA. Exclusive prefix sums of the three counts in frame order: feature rows, point rows and (append mode)
//                         key-frame rows are handed out frame by frame.
//   commit_write_kernel : one CTA per frame. bad = 1 for every matched point whose count ended <= 0; then the key frame: its row, the
//                         matches and the new corners as feature rows, the new points (found 1). Every observing feature row is pushed
//                         onto its point's last_obs with atomicExch, the replaced row kept in a scratch link; the push order is
//                         arbitrary, the set of rows a point collects is not.
//   commit_link_kernel  : one CTA per frame. For each point the feature whose push replaced an old row (or -1) owns the pushed rows: it
//                         orders them newest first above the old chain -- the chain dsdtm_store_append_keyframe's store_link_kernel builds
//                         when the key frames are appended one by one in frame order. Rows grow in frame order, so newest = largest row.
//                         The owner merge-sorts the list: O(k log k) dependent loads on one thread for a point that k key frames of one
//                         commit observe (k = 1 when every map has at most one frame per step; k = frames per map when a map serves
//                         several frames of the step).
#include "ctx.cuh"
#include "se3_exact.cuh"

namespace dsdtm {

namespace {

static const int kCmThreads = 256;

struct CommitArgs {
    int n, kf;                                  // frames; 1 when the run had flags bit 3 (key frames)
    double thr;
    const int* nm; const dsdtm_match* match; const dsdtm_ba_obs* obs; const double* res; const double* pose; const int* cur_slots;
    const uint8_t* want; const int* nnew; const dsdtm_corner* corners; const dsdtm_lifted* lifted; int stride;
    const int* kf_rows;                         // reserved rows per frame or null (append)
    int k0, f0, p0;                             // table sizes before the commit
    dsdtm_store_kf* kfs; dsdtm_store_feat* feats; dsdtm_store_point* pts; int* found;
    int* cnt;                                   // 3n: feature rows, new points, key frame per frame
    int* out;                                   // 5n: kf_row, point_first, n_points, feat_first, n_feats; then 4 totals
    int* push;                                  // per new feature row: the row its chain push replaced
};

__global__ void __launch_bounds__(kCmThreads) commit_found_kernel(const CommitArgs a)
{
    const int f = blockIdx.x, t = threadIdx.x;
    const int nm = a.nm[f];
    if (nm < 0) {                                                    // candidate overflow: the frame changes nothing
        if (t == 0) { a.cnt[f] = 0; a.cnt[a.n + f] = 0; a.cnt[2 * a.n + f] = 0; }
        return;
    }
    for (int m = t; m < nm; m += kCmThreads) {
        const size_t i = (size_t)f * DSDTM_TRACK_MAX_MATCHES + m;
        const int p = a.match[i].point;
        const int d = (a.res[i] > a.thr && !a.pts[p].bad) ? 0 : 1;   // IncreaseFound, then EraseFound (strict '>', ref: :81-94)
        if (d) atomicAdd(a.found + p, d);
    }
    const bool kf = a.kf && a.want[f];
    int n_pts = 0, n_new = 0;
    if (kf) {
        n_new = a.nnew[f];
        for (int j0 = 0; j0 < n_new; j0 += kCmThreads) {
            const int j = j0 + t;
            n_pts += __syncthreads_count(j < n_new && a.lifted[(size_t)f * a.stride + j].status == DSDTM_LIFT_OK);
        }
    }
    if (t == 0) { a.cnt[f] = kf ? nm + n_new : 0; a.cnt[a.n + f] = n_pts; a.cnt[2 * a.n + f] = kf ? 1 : 0; }
}

__global__ void __launch_bounds__(1024) commit_scan_kernel(const CommitArgs a)
{
    __shared__ int s_w[3][32];
    __shared__ int s_carry[4];
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t < 4) s_carry[t] = 0;
    __syncthreads();
    for (int f0 = 0; f0 < a.n; f0 += 1024) {
        const int f = f0 + t;
        const bool in = f < a.n;
        int v[3], x[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            v[q] = in ? a.cnt[q * a.n + f] : 0;
            x[q] = v[q];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x[q], o); if (lane >= o) x[q] += y; }
            if (lane == 31) s_w[q][warp] = x[q];
        }
        __syncthreads();
        if (warp == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                int w = s_w[q][lane];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w += y; }
                s_w[q][lane] = w;                                    // inclusive over warps
            }
        }
        __syncthreads();
        int off[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) off[q] = s_carry[q] + (warp ? s_w[q][warp - 1] : 0) + x[q] - v[q];
        if (in) {
            const bool kf = v[2] != 0;
            a.out[f] = kf ? (a.kf_rows ? a.kf_rows[f] : a.k0 + off[2]) : -1;
            a.out[a.n + f] = kf ? a.p0 + off[1] : -1;
            a.out[2 * a.n + f] = v[1];
            a.out[3 * a.n + f] = a.f0 + off[0];
            a.out[4 * a.n + f] = v[0];
        }
        const int fmax = __reduce_max_sync(0xffffffffu, (unsigned)(in && v[2] ? v[0] : 0));
        __syncthreads();
        if (t == 0) {
#pragma unroll
            for (int q = 0; q < 3; ++q) s_carry[q] += s_w[q][31];
        }
        if (lane == 0) atomicMax(s_carry + 3, fmax);
        __syncthreads();
    }
    if (t < 4) a.out[5 * a.n + t] = s_carry[t];
}

__global__ void __launch_bounds__(kCmThreads) commit_write_kernel(const CommitArgs a)
{
    __shared__ int s_wcnt[kCmThreads / 32];
    const int f = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int nm = a.nm[f];
    if (nm < 0) return;
    const dsdtm_match* M = a.match + (size_t)f * DSDTM_TRACK_MAX_MATCHES;
    for (int m = t; m < nm; m += kCmThreads) {
        const int p = M[m].point;
        if (a.found[p] <= 0) a.pts[p].bad = 1;                       // ref: MapPoint::EraseFound
    }
    const int r = a.out[f];
    if (r < 0) return;                                               // no key frame: the whole CTA leaves
    const int fb = a.out[3 * a.n + f], nf = a.out[4 * a.n + f], pb = a.out[a.n + f];
    const dsdtm_ba_obs* O = a.obs + (size_t)f * DSDTM_TRACK_MAX_MATCHES;
    for (int m = t; m < nm; m += kCmThreads) {                       // the matches first (mvFeatures order)
        const dsdtm_match mt = M[m];
        dsdtm_store_feat o;
        o.mp = mt.point; o.level = mt.level; o.px[0] = mt.px[0]; o.px[1] = mt.px[1];
#pragma unroll
        for (int k = 0; k < 3; ++k) o.normal[k] = O[m].normal[k];   // Frame::Add_Feature's bearing, as PoseOptimization saw it
        o.is_obs = r + 1; o.next_obs = -1;
        a.feats[fb + m] = o;
    }
    const int n_new = nf - nm;
    int base = 0;
    for (int j0 = 0; j0 < n_new; j0 += kCmThreads) {                 // then the new corners, a new point for each one with a depth
        const int j = j0 + t;
        const dsdtm_lifted* L = a.lifted + (size_t)f * a.stride;
        const bool ok = j < n_new && L[j].status == DSDTM_LIFT_OK;
        const unsigned bal = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) s_wcnt[warp] = __popc(bal);
        __syncthreads();
        int off = 0, tot = 0;
#pragma unroll
        for (int w = 0; w < kCmThreads / 32; ++w) { const int c = s_wcnt[w]; off += w < warp ? c : 0; tot += c; }
        if (j < n_new) {
            const dsdtm_lifted l = L[j];
            const int p = ok ? pb + base + off + __popc(bal & ((1u << lane) - 1u)) : -1;
            dsdtm_store_feat o;
            o.mp = p; o.level = a.corners[(size_t)f * a.stride + j].level; o.px[0] = l.px[0]; o.px[1] = l.px[1];
#pragma unroll
            for (int k = 0; k < 3; ++k) o.normal[k] = l.normal[k];
            o.is_obs = ok ? r + 1 : 0; o.next_obs = -1;
            a.feats[fb + nm + j] = o;
            if (ok) {
                dsdtm_store_point q;
                q.point_w[0] = l.point_w[0]; q.point_w[1] = l.point_w[1]; q.point_w[2] = l.point_w[2];
                q.bad = 0; q.last_obs = -1;
                a.pts[p] = q;
                a.found[p] = 1;                                      // MapPoint's constructor
            }
        }
        base += tot;
        __syncthreads();
    }
    if (t == 0) {
        dsdtm_store_kf k;
        const double* P = a.pose + 7 * (size_t)f;
        double inv[7];
        se3_inv_exact(P, inv);                                       // KeyFrame::Get_CameraCnt()
        k.slot = a.cur_slots[f]; k.feat_begin = fb; k.feat_count = nf; k.reserved = 0;
#pragma unroll
        for (int q = 0; q < 7; ++q) k.pose_c2w[q] = P[q];
#pragma unroll
        for (int q = 0; q < 3; ++q) k.center[q] = inv[4 + q];
        a.kfs[r] = k;
    }
    __syncthreads();                                                 // the new points exist before their chains are pushed
    for (int j = t; j < nf; j += kCmThreads) {
        const dsdtm_store_feat& o = a.feats[fb + j];
        if (o.is_obs) a.push[fb + j - a.f0] = atomicExch(&a.pts[o.mp].last_obs, fb + j);
    }
}

__global__ void __launch_bounds__(kCmThreads) commit_link_kernel(const CommitArgs a)
{
    const int f = blockIdx.x;
    const int r = a.out[f];
    if (r < 0) return;
    const int fb = a.out[3 * a.n + f], nf = a.out[4 * a.n + f];
    for (int j = threadIdx.x; j < nf; j += kCmThreads) {
        const int g = fb + j;
        if (!a.feats[g].is_obs || a.push[g - a.f0] >= a.f0) continue;     // not the owner of its point's pushes
        const int p = a.feats[g].mp;
        // the pushed rows (push links, newest push first) end at the point's chain before the commit (or -1). They are threaded into a
        // list through next_obs, which only this thread writes for them, and merge-sorted by descending row: O(k log k) for k rows
        int x = a.pts[p].last_obs, head = -1, prev = -1;
        while (x >= a.f0) {
            if (prev < 0) head = x; else a.feats[prev].next_obs = x;
            prev = x;
            x = a.push[x - a.f0];
        }
        a.feats[prev].next_obs = -1;
        const int old = x;                                           // the chain the point had before the commit
        int tail = -1;
        for (int run = 1;; run *= 2) {                               // bottom-up merge sort of a linked list, stable, no extra memory
            int l = head, merges = 0;
            head = -1; tail = -1;
            while (l >= 0) {
                ++merges;
                int q = l, nl = 0;
                for (int i = 0; i < run && q >= 0; ++i) { ++nl; q = a.feats[q].next_obs; }
                int nr = run;
                while (nl > 0 || (nr > 0 && q >= 0)) {
                    int e;
                    if (nl > 0 && (nr == 0 || q < 0 || l > q)) { e = l; l = a.feats[l].next_obs; --nl; }
                    else { e = q; q = a.feats[q].next_obs; --nr; }
                    if (tail < 0) head = e; else a.feats[tail].next_obs = e;
                    tail = e;
                }
                l = q;
            }
            a.feats[tail].next_obs = -1;
            if (merges <= 1) break;
        }
        a.feats[tail].next_obs = old;                                // above the chain the point had before the commit
        a.pts[p].last_obs = head;
    }
}

}  // namespace

cudaError_t launch_store_commit(dsdtm_ctx* c, const StoreCommitArgs& s, cudaStream_t st)
{
    const auto& b = c->batch;
    CommitArgs a;
    a.n = b.n_pairs; a.kf = s.keyframes ? 1 : 0; a.thr = (double)s.threshold;
    a.nm = c->trk_nobs_d; a.match = c->trk_match_d; a.obs = c->trk_obs_d; a.res = c->trk_res_d; a.pose = c->trk_pose_out_d;
    a.cur_slots = c->cur_slots_d;
    a.want = c->kf_want_d; a.nnew = c->kf_nnew_d; a.corners = c->kf_corner_d; a.lifted = c->kf_lifted_d; a.stride = b.kf_max_fts;
    a.kf_rows = s.kf_rows_d;
    a.k0 = (int)c->st_kfs_n; a.f0 = (int)c->st_feats_n; a.p0 = (int)c->st_pts_n;
    a.kfs = c->st_kfs_d; a.feats = c->st_feats_d; a.pts = c->st_pts_d; a.found = c->st_found_d;
    a.cnt = s.cnt_d; a.out = s.out_d; a.push = s.push_d;
    commit_found_kernel<<<a.n, kCmThreads, 0, st>>>(a);
    commit_scan_kernel<<<1, 1024, 0, st>>>(a);
    commit_write_kernel<<<a.n, kCmThreads, 0, st>>>(a);
    commit_link_kernel<<<a.n, kCmThreads, 0, st>>>(a);
    c->launches += 4;
    return cudaGetLastError();
}

}  // namespace dsdtm
