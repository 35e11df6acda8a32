// select.cu -- Feature_Alignment::SearchLocalPoints' greedy selection (ref: src/Feature_alignment.cpp:71-121) over the records of the
// batched refinement chain, and the Optimizer::PoseOptimization inputs it hands to pose_opt.cu without a host round trip.
//
//   track_select_kernel : one warp per frame pair, four pairs per CTA:
//     1. compaction  : the pair's eligible records -- in a cell, OBS_OK | REF_OK, aligned (level >= 0), CONVERGED -- as 64-bit keys
//                      (cell << 42 | ~found << 10 | j). Every other record is skipped by the reference whatever the mask holds, so
//                      it never needs a mask test (the NaN projections of Q3 are never CONVERGED and never reach cvRound).
//     2. order       : rank of each key by counting (the keys are distinct: j is in them) = cells ascending, found descending, j
//                      ascending -- std::list::sort is stable and the insertion order of the chain's cells is j.
//     3. walk        : 32 candidates at a time in that order. Each lane tests its candidate against the circles painted so far
//                      (mask(cvRound((float)px_proj)) != 255); then the first alive lane wins its cell, broadcasts its circle
//                      centre, and the lanes behind it drop out when they share its cell or fall inside the new circle.
//     4. records     : per match (mvFeatures order) the dsdtm_ba_obs of Frame::Add_Feature: bearing of the float px, the staged
//                      feature's point, the search level; the match count; cur.Get_Pose() = T_c2r * T_ref for the solve.
// The mask is never materialised (38-45 KB per pair would cap residency): a pixel is painted iff some earlier centre lies within
// |dy| <= r and |dx| <= span[|dy|], where span is the half-width of cv::circle(.., -1)'s row dy (OpenCV's midpoint routine). The
// tested pixel is inside the image (IsInImage(px, 8) put it in a cell), so the clipping at the image border changes nothing.
#include <algorithm>

#include "ctx.cuh"
#include "se3_exact.cuh"

namespace dsdtm {

namespace {

static const int kSelWarps = 4;
static const int kMaxRadius = 64;                 // Camera.CellSize bound of the span table
static const int kCap = DSDTM_TRACK_MAX_MATCHES;

struct SelArgs {
    const dsdtm_reproj* rec; const int* found; const dsdtm_ref_feat* feats; int feat_stride;
    const double* poses_c2r; const double* poses_ref;
    int n_pairs, ppp, per_warp;                   // per_warp = 8-byte words of shared memory per warp
    // store mode: records sb_rec (ppp per frame, the first n_cand valid, in order), found per store point row, points from the store
    const dsdtm_store_cand* srec; const int* n_cand; const dsdtm_store_point* pts; int n_found; const double* pose10; int jbits;
    float fx, fy, cx, cy;
    int radius; int span[kMaxRadius + 1];
    dsdtm_match* match; dsdtm_ba_obs* obs; int* n_match; double* pose_in;
};

__device__ __forceinline__ bool in_circle(int x, int y, int cx, int cy, int r, const int* span)
{
    const long long dy = llabs((long long)y - cy), dx = llabs((long long)x - cx);
    return dy <= r && dx <= span[dy];
}

// kStore: the records are the store-backed chain's (dsdtm_batch_stage_store): j is the record index, which is the order of ReprojectPoint;
// found comes from the point's row, the match names the store point, and a frame whose candidates overflowed its rows gets n_match -1
template <bool kStore>
__global__ void __launch_bounds__(kSelWarps * 32) track_select_kernel(const SelArgs a)
{
    extern __shared__ unsigned long long sel_smem[];
    __shared__ int s_span[kMaxRadius + 1];
    for (int k = threadIdx.x; k <= a.radius; k += blockDim.x) s_span[k] = a.span[k];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int pair = blockIdx.x * kSelWarps + warp;
    if (pair >= a.n_pairs) return;                // whole warps leave; no CTA-wide barrier follows
    unsigned long long* key = sel_smem + (size_t)warp * a.per_warp;
    int2* circ = reinterpret_cast<int2*>(key + a.ppp);
    int* order = reinterpret_cast<int*>(circ + kCap);
    const dsdtm_reproj* R = a.rec + (size_t)pair * a.ppp;
    const dsdtm_store_cand* SR = a.srec + (size_t)pair * a.ppp;
    const int* F = a.found + (size_t)pair * a.ppp;
    const int jb = kStore ? a.jbits : 10;
    int n_rec = a.ppp;
    bool overflow = false;
    if (kStore) { const int nc = a.n_cand[pair]; overflow = nc > a.ppp; n_rec = overflow ? 0 : nc; }

    // 1. compaction in j order
    int n = 0;
    for (int j0 = 0; j0 < n_rec; j0 += 32) {
        const int j = j0 + lane;
        bool ok = false;
        unsigned long long k = 0;
        if (j < n_rec) {
            const dsdtm_reproj& rj = kStore ? SR[j].r : R[j];
            const int need = DSDTM_LM_OBS_OK | DSDTM_LM_REF_OK | DSDTM_LM_CONVERGED;
            const int cell = rj.cell;
            ok = cell >= 0 && (rj.flags & need) == need && rj.level >= 0;
            int fc = 1;                                                     // a point appended after staging: MapPoint::mnFound starts at 1
            if (!kStore) fc = F[j];
            else if (SR[j].mp < a.n_found) fc = a.found[SR[j].mp];
            const unsigned fdesc = ~((unsigned)fc ^ 0x80000000u);           // found descending as an unsigned ascending key
            k = ((unsigned long long)(unsigned)cell << (32 + jb)) | ((unsigned long long)fdesc << jb) | (unsigned)j;
        }
        const unsigned b = __ballot_sync(0xffffffffu, ok);
        if (ok) key[n + __popc(b & ((1u << lane) - 1u))] = k;
        n += __popc(b);
    }
    __syncwarp();
    // 2. the reference's visiting order
    for (int e = lane; e < n; e += 32) {
        const unsigned long long k = key[e];
        int rank = 0;
        for (int q = 0; q < n; ++q) rank += key[q] < k ? 1 : 0;
        order[rank] = (int)(k & ((1u << jb) - 1u));
    }
    __syncwarp();
    // 3. the greedy walk
    dsdtm_match* M = a.match + (size_t)pair * kCap;
    int n_match = 0, won_cell = -1;
    for (int b0 = 0; b0 < n && n_match < kCap; b0 += 32) {
        const int e = b0 + lane;
        bool alive = e < n;
        int j = 0, cell = -1, x = 0, y = 0, mx = 0, my = 0, level = 0;
        float p0 = 0.f, p1 = 0.f;
        if (alive) {
            j = order[e];
            const dsdtm_reproj& r = kStore ? SR[j].r : R[j];
            cell = r.cell; level = r.level;
            x = __float2int_rn(__double2float_rn(r.px_proj[0])); y = __float2int_rn(__double2float_rn(r.px_proj[1]));   // Mat::at(cvRound)
            p0 = __double2float_rn(r.px[0]); p1 = __double2float_rn(r.px[1]);                                             // Point2f(px)
            mx = __float2int_rn(p0); my = __float2int_rn(p1);                                                             // cv::Point(Point2f)
            alive = cell != won_cell;
            for (int q = 0; q < n_match && alive; ++q) alive = !in_circle(x, y, circ[q].x, circ[q].y, a.radius, s_span);
        }
        while (n_match < kCap) {
            const unsigned bal = __ballot_sync(0xffffffffu, alive);
            if (!bal) break;
            const int w = __ffs(bal) - 1;
            const int wcell = __shfl_sync(0xffffffffu, cell, w), wx = __shfl_sync(0xffffffffu, mx, w), wy = __shfl_sync(0xffffffffu, my, w);
            if (lane == w) {
                circ[n_match] = make_int2(mx, my);
                dsdtm_match m; m.point = kStore ? SR[j].mp : j; m.px[0] = p0; m.px[1] = p1; m.level = level;
                M[n_match] = m;
            }
            ++n_match; won_cell = wcell;
            if (lane <= w || cell == wcell) alive = false;
            else if (alive && in_circle(x, y, wx, wy, a.radius, s_span)) alive = false;
        }
        __syncwarp();
    }
    // 4. PoseOptimization's inputs
    dsdtm_ba_obs* O = a.obs + (size_t)pair * kCap;
    const dsdtm_ref_feat* Fe = a.feats + (size_t)pair * a.feat_stride;
    for (int m = lane; m < n_match; m += 32) {
        const dsdtm_match mt = M[m];
        dsdtm_ba_obs o;
        feature_normal_exact(mt.px[0], mt.px[1], a.fx, a.fy, a.cx, a.cy, o.normal);                   // ref: src/Frame.cpp:83-92
#pragma unroll
        for (int k = 0; k < 3; ++k) o.point_w[k] = kStore ? a.pts[mt.point].point_w[k] : Fe[mt.point].point_w[k];
        o.level = mt.level; o.reserved = 0;
        O[m] = o;
    }
    if (kStore && lane == 0) {
        a.n_match[pair] = overflow ? -1 : n_match;
#pragma unroll
        for (int k = 0; k < 7; ++k) a.pose_in[7 * (size_t)pair + k] = a.pose10[10 * (size_t)pair + k];   // composed by the prelude
    } else if (lane == 0) {
        a.n_match[pair] = n_match;
        double Tc2r[7], Tr[7], pc[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) { Tc2r[k] = a.poses_c2r[7 * (size_t)pair + k]; Tr[k] = a.poses_ref[7 * (size_t)pair + k]; }
        se3_mul_exact(Tc2r, Tr, pc);                                                                   // ref: src/Sprase_ImageAlign.cpp:57
#pragma unroll
        for (int k = 0; k < 7; ++k) a.pose_in[7 * (size_t)pair + k] = pc[k];
    }
}

// bits of an index below n (at least 1)
int index_bits(int n)
{
    int b = 1;
    while ((1 << b) < n) ++b;
    return b;
}

SelArgs select_args(dsdtm_ctx* c, int n_pairs, int ppp)
{
    SelArgs a;
    a.rec = c->pair_reproj_d; a.found = c->trk_found_d; a.feats = c->feats_d; a.feat_stride = 0;
    a.poses_c2r = c->poses_out_d; a.poses_ref = c->poses_ref_d;
    a.srec = nullptr; a.n_cand = nullptr; a.pts = nullptr; a.n_found = 0; a.pose10 = nullptr; a.jbits = 10;
    a.n_pairs = n_pairs; a.ppp = ppp;
    a.per_warp = ppp + kCap + (ppp + 1) / 2;      // keys, circle centres, order
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    // row half-widths of cv::circle(img, c, r, color, -1) (OpenCV drawing.cpp, the filled midpoint circle)
    const int r = c->prm.cell_size;
    a.radius = (r < 0 || r > kMaxRadius) ? -1 : r;       // refused by the launchers
    if (a.radius < 0) return a;
    for (int k = 0; k <= kMaxRadius; ++k) a.span[k] = -1;
    {
        int err = 0, dx = r, dy = 0, plus = 1, minus = (r << 1) - 1;
        while (dx >= dy) {
            a.span[dy] = std::max(a.span[dy], dx);
            a.span[dx] = std::max(a.span[dx], dy);
            dy++;
            err += plus;
            plus += 2;
            const int mask = (err <= 0) - 1;
            err -= minus & mask;
            dx += mask;
            minus -= mask & 2;
        }
    }
    a.match = c->trk_match_d; a.obs = c->trk_obs_d; a.n_match = c->trk_nobs_d; a.pose_in = c->trk_pose_in_d;
    return a;
}

}  // namespace

size_t track_select_smem(int ppp) { return (size_t)kSelWarps * (ppp + kCap + (ppp + 1) / 2) * sizeof(unsigned long long); }

cudaError_t launch_track_select(dsdtm_ctx* c, int n_pairs, int feat_stride, int ppp, cudaStream_t s)
{
    SelArgs a = select_args(c, n_pairs, ppp);
    a.feat_stride = feat_stride;
    if (a.radius < 0) return cudaErrorInvalidValue;
    track_select_kernel<false><<<(n_pairs + kSelWarps - 1) / kSelWarps, kSelWarps * 32, track_select_smem(ppp), s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_track_select_store(dsdtm_ctx* c, int n_pairs, int cpf, const int* found_d, int n_found, cudaStream_t s)
{
    SelArgs a = select_args(c, n_pairs, cpf);
    if (a.radius < 0) return cudaErrorInvalidValue;
    a.srec = c->sb_rec_d; a.n_cand = c->sb_ncand_d; a.pts = c->st_pts_d; a.pose10 = c->sb_pose10_d;
    a.found = found_d; a.n_found = n_found;
    a.jbits = index_bits(cpf);
    track_select_kernel<true><<<(n_pairs + kSelWarps - 1) / kSelWarps, kSelWarps * 32, track_select_smem(cpf), s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

int track_select_key_bits(const dsdtm_ctx* c, int ppp) { return index_bits(c->n_cells) + 32 + index_bits(ppp); }

cudaError_t track_select_init(dsdtm_ctx* c)
{
    int max_smem = 0;
    cudaError_t e = cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(track_select_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem - 1024);
    return e;
}

int track_select_max_radius() { return kMaxRadius; }

}  // namespace dsdtm
