// capi.cu -- the extern "C" boundary (include/dsdtm_gpu.h): context, HBM pools, staging, launches, CUDA-graph replay.
// No compute happens on the host here; if the CUDA device / kernels are unavailable every entry point fails loudly.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "ctx.cuh"

namespace dsdtm {

int build_fast_tiles(const LevelGeom& g, int* out, int* level_first);

static std::string g_create_error;

void stage_begin(dsdtm_ctx* c, int stage)
{
    if (!c->profiling) return;
    StageTimer& t = c->timer;
    if (t.n >= StageTimer::kMaxEv) stage_collect(c);
    t.stage[t.n] = stage;
    cudaEventRecord(t.ev0[t.n], c->stream);
}

void stage_end(dsdtm_ctx* c, int n_launches)
{
    if (!c->profiling) return;
    StageTimer& t = c->timer;
    cudaEventRecord(t.ev1[t.n], c->stream);
    t.launches[t.stage[t.n]] += n_launches;
    t.n++;
}

int stage_collect(dsdtm_ctx* c)
{
    StageTimer& t = c->timer;
    if (t.n == 0) return 0;
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < t.n; ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, t.ev0[i], t.ev1[i]);
        t.ms[t.stage[i]] += ms;
    }
    t.n = 0;
    return 0;
}

template <class T>
static int dalloc(dsdtm_ctx* c, T** p, size_t n)
{
    cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T));
    if (e != cudaSuccess) return fail(c, DSDTM_E_NOMEM, "cudaMalloc", e);
    return 0;
}

template <class T>
static int grow(dsdtm_ctx* c, T** p, size_t* cap, size_t n)
{
    if (n <= *cap) return 0;
    if (*p) { cudaFree(*p); *p = nullptr; *cap = 0; }
    const size_t want = std::max<size_t>(n + n / 2, 256);
    if (dalloc(c, p, want)) return DSDTM_E_NOMEM;
    *cap = want;
    return 0;
}

// grow() for tables whose contents must survive: the first `keep` elements are copied to the new allocation
template <class T>
static int grow_keep(dsdtm_ctx* c, T** p, size_t* cap, size_t n, size_t keep)
{
    if (n <= *cap) return 0;
    T* old = *p;
    T* fresh = nullptr;
    const size_t want = std::max<size_t>(2 * n, 1024);
    if (dalloc(c, &fresh, want)) return DSDTM_E_NOMEM;
    if (old && keep) {
        cudaError_t e = cudaMemcpyAsync(fresh, old, keep * sizeof(T), cudaMemcpyDeviceToDevice, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) { cudaFree(fresh); return fail(c, DSDTM_E_CUDA, "table copy", e); }
    }
    if (old) cudaFree(old);
    *p = fresh; *cap = want;
    return 0;
}

static int ensure_pinned(dsdtm_ctx* c, size_t bytes)
{
    if (bytes <= c->pinned_bytes) return 0;
    if (c->pinned) cudaFreeHost(c->pinned);
    c->pinned = nullptr; c->pinned_bytes = 0;
    cudaError_t e = cudaMallocHost((void**)&c->pinned, bytes);
    if (e != cudaSuccess) return fail(c, DSDTM_E_NOMEM, "cudaMallocHost", e);
    c->pinned_bytes = bytes;
    return 0;
}

// Small synchronous calls (one frame, a few hundred features / patches) are dominated by driver overhead when their inputs
// and outputs are pageable host buffers: every cudaMemcpyAsync on pageable memory is staged and synchronised by the driver
// (~8 us each, 8-10 per call). The Stager bounces them through a fixed pinned arena instead: inputs are memcpy'd into it and
// copied from there (truly asynchronous, ~2 us per call), outputs land in it and are handed out after the one stream
// synchronisation. Calls whose buffers do not fit use the caller's pointers directly (large batches should pass pinned
// memory from dsdtm_host_alloc anyway).
static const size_t kStageBytes = 1u << 20;
struct Stager {
    dsdtm_ctx* c;
    size_t off = 0;
    bool active;
    struct Out { void* dst; const void* src; size_t bytes; } outs[8];
    int n_outs = 0;
    Stager(dsdtm_ctx* ctx, size_t total_bytes) : c(ctx), active(ctx->stage_pin != nullptr && total_bytes + 16 * 16 <= kStageBytes) {}
    uint8_t* carve(size_t bytes) { uint8_t* p = c->stage_pin + off; off += (bytes + 15) & ~(size_t)15; return p; }
    const void* in(const void* src, size_t bytes)
    {
        if (!active || bytes == 0) return src;
        uint8_t* p = carve(bytes);
        std::memcpy(p, src, bytes);
        return p;
    }
    void* out(void* dst, size_t bytes)
    {
        if (!active || bytes == 0 || n_outs == 8) return dst;
        uint8_t* p = carve(bytes);
        outs[n_outs++] = Out{ dst, p, bytes };
        return p;
    }
    void finish() { for (int i = 0; i < n_outs; ++i) std::memcpy(outs[i].dst, outs[i].src, outs[i].bytes); }   // after the stream sync
};

// The two calls made once per tracked frame (dsdtm_sparse_align, dsdtm_align2d_batch) go one step further: all inputs are
// packed into the pinned arena and travel in ONE host-to-device copy into its device mirror, the kernels read and write the
// mirror directly (the context's staging pointers are swapped for the duration of the launch), and all outputs come back in
// ONE device-to-host copy. 6 + 2..4 serialised DMA operations per call become 1 + 1.
struct Arena {
    dsdtm_ctx* c;
    size_t in_off = 0, out_off = 0, out_end = 0;
    bool active;
    struct Out { void* dst; size_t off; size_t bytes; } outs[8];
    int n_outs = 0;
    static size_t pad(size_t b) { return (b + 15) & ~(size_t)15; }
    Arena(dsdtm_ctx* ctx, size_t in_bytes, size_t out_bytes, int n_in, int n_out)
        : c(ctx), active(ctx->stage_pin && ctx->stage_dev && in_bytes + out_bytes + 16 * (size_t)(n_in + n_out) + 512 <= kStageBytes)
    {
        out_off = out_end = (in_bytes + 16 * (size_t)n_in + 255) & ~(size_t)255;
    }
    template <class T> T* in(const T* src, size_t n)                 // copies n elements into the arena, returns the DEVICE address
    {
        const size_t o = in_off;
        std::memcpy(c->stage_pin + o, src, n * sizeof(T));
        in_off += pad(n * sizeof(T));
        return reinterpret_cast<T*>(c->stage_dev + o);
    }
    template <class T> T* in_fill(size_t n, T** host)                // same, but the caller fills the host side itself
    {
        const size_t o = in_off;
        *host = reinterpret_cast<T*>(c->stage_pin + o);
        in_off += pad(n * sizeof(T));
        return reinterpret_cast<T*>(c->stage_dev + o);
    }
    template <class T> T* out(T* dst, size_t n)                      // reserves an output range, returns the DEVICE address
    {
        const size_t o = out_end;
        out_end += pad(n * sizeof(T));
        if (dst) outs[n_outs++] = Out{ dst, o, n * sizeof(T) };
        return reinterpret_cast<T*>(c->stage_dev + o);
    }
    template <class T> const T* host_view(const T* dev) const { return reinterpret_cast<const T*>(c->stage_pin + (reinterpret_cast<const uint8_t*>(dev) - c->stage_dev)); }
    cudaError_t upload(cudaStream_t s) { return cudaMemcpyAsync(c->stage_dev, c->stage_pin, in_off, cudaMemcpyHostToDevice, s); }
    cudaError_t download(cudaStream_t s)
    {
        return cudaMemcpyAsync(c->stage_pin + out_off, c->stage_dev + out_off, out_end - out_off, cudaMemcpyDeviceToHost, s);
    }
    void finish() { for (int i = 0; i < n_outs; ++i) std::memcpy(outs[i].dst, c->stage_pin + outs[i].off, outs[i].bytes); }
};
template <class T> struct PtrSwap {     // points a context staging pointer at the arena for the duration of a launch
    T*& ref; T* saved;
    PtrSwap(T*& r, T* v) : ref(r), saved(r) { r = v; }
    ~PtrSwap() { ref = saved; }
};

static void decode_cells(const dsdtm_ctx* c, const unsigned long long* keys, float seed, dsdtm_corner* out, int n)
{
    for (int i = 0; i < n; ++i) {
        const unsigned long long k = keys[i];
        if (k == 0) { out[i] = dsdtm_corner{ 0, 0, 0, seed }; continue; }    // ref: src/Feature_detection.cpp:74
        const unsigned order = ~(unsigned)(k & 0xFFFFFFFFull);
        const unsigned bits = (unsigned)(k >> 32);
        float s; std::memcpy(&s, &bits, 4);
        const int L = order >> 28, y = (order >> 14) & 0x3FFF, x = order & 0x3FFF;
        out[i] = dsdtm_corner{ x << L, y << L, L, s };                       // ref: :106
    }
}

// every captured step of dsdtm_batch_run: after anything a graph has baked into its launch arguments changes
static void drop_graphs(dsdtm_ctx* c)
{
    for (cudaGraphExec_t& g : c->batch.graph)
        if (g) { cudaGraphExecDestroy(g); g = nullptr; }
}

// a map-store change: a captured store-backed step has the tables, their sizes and the grids derived from them baked in (the tables may
// have been reallocated); steps of the other modes never read the store and stay captured
static void drop_store_graphs(dsdtm_ctx* c)
{
    if (c->batch.store_staged) drop_graphs(c);
}

static int check_slot(dsdtm_ctx* c, int slot, int n = 1)
{
    if (slot < 0 || n < 0 || slot + n > c->prm.max_frames) return fail(c, DSDTM_E_ARG, "frame slot out of range");
    return 0;
}

// the pyramid, FAST, CLAHE and key-frame lift kernels take the frame / pair index from gridDim.y or gridDim.z (at most 65535);
// checked before anything is enqueued, so that a refused call leaves no partial work behind
static int check_grid_frames(dsdtm_ctx* c, int n)
{
    if (n > DSDTM_MAX_BATCH_FRAMES) return fail(c, DSDTM_E_ARG, "more than DSDTM_MAX_BATCH_FRAMES frames or pairs in one batched call");
    return 0;
}

}  // namespace dsdtm

using namespace dsdtm;

extern "C" {

int dsdtm_abi_version(void) { return DSDTM_ABI_VERSION; }
const char* dsdtm_create_error(void) { return g_create_error.c_str(); }

dsdtm_ctx* dsdtm_create(int device, const dsdtm_cam* cam, const dsdtm_params* prm)
{
    g_create_error.clear();
    if (!cam || !prm) { g_create_error = "null cam/params"; return nullptr; }
    if (prm->levels < 1 || prm->levels > DSDTM_MAX_LEVELS || cam->width < 8 || cam->height < 8 || cam->width > 16383 ||
        cam->height > 16383 || prm->cell_size < 1 || prm->max_feats < 1 || prm->max_feats > DSDTM_MAX_FEATS_LIMIT ||
        prm->max_frames < 1 || prm->max_batch < 1 || prm->max_patches < 0) {
        g_create_error = "bad cam/params";
        return nullptr;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e);
        return nullptr;
    }
    if (device < 0 || device >= ndev) { g_create_error = "device index out of range"; return nullptr; }
    if ((e = cudaSetDevice(device)) != cudaSuccess) { g_create_error = cudaGetErrorString(e); return nullptr; }

    dsdtm_ctx* c = new dsdtm_ctx();
    c->device = device; c->cam = *cam; c->prm = *prm;
    cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);

    // level geometry: dense levels, 16-byte aligned offsets, >= 64 bytes of zero padding at the end of a slot
    LevelGeom& g = c->geo;
    g.levels = prm->levels;
    unsigned off = 0;
    for (int l = 0; l < g.levels; ++l) {
        g.w[l] = l ? (g.w[l - 1] + 1) / 2 : cam->width;
        g.h[l] = l ? (g.h[l - 1] + 1) / 2 : cam->height;
        g.off[l] = off;
        off += (unsigned)g.w[l] * g.h[l];
        off = (off + 15u) & ~15u;
    }
    for (int l = g.levels; l < DSDTM_MAX_LEVELS; ++l) { g.w[l] = g.h[l] = 0; g.off[l] = off; }
    g.frame_stride = (off + 64u + 255u) & ~255u;
    c->grid_rows = (cam->height + prm->cell_size - 1) / prm->cell_size;     // ref: src/Feature_detection.cpp:18-19 (ceil)
    c->grid_cols = (cam->width + prm->cell_size - 1) / prm->cell_size;
    c->n_cells = c->grid_rows * c->grid_cols;

    auto bail = [&](const char* what) -> dsdtm_ctx* {
        g_create_error = std::string(what) + ": " + c->err;
        dsdtm_destroy(c);
        return nullptr;
    };
#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { c->err = cudaGetErrorString(e__); return bail(#call); } } while (0)
    CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->copy_stream[0], cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&c->copy_stream[1], cudaStreamNonBlocking));
    CK(cudaEventCreate(&c->ev_a));
    CK(cudaEventCreate(&c->ev_b));
    CK(cudaEventCreate(&c->ev_t0));
    CK(cudaEventCreate(&c->ev_t1));
    CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    for (int i = 0; i < kMaxStepStreams; ++i) {
        CK(cudaStreamCreateWithFlags(&c->step_stream[i], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 4; ++i) CK(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
    for (int i = 0; i < 8; ++i) { CK(cudaEventCreateWithFlags(&c->ev_up[i], cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&c->ev_done[i], cudaEventDisableTiming)); }
    for (int i = 0; i < StageTimer::kMaxEv; ++i) { CK(cudaEventCreate(&c->timer.ev0[i])); CK(cudaEventCreate(&c->timer.ev1[i])); }

    const size_t B = prm->max_batch, F = prm->max_feats, P = std::max(prm->max_patches, 1);
    const size_t pool = (size_t)prm->max_frames * g.frame_stride;
    if (dalloc(c, &c->frames_d, pool)) return bail("frame pool");
    CK(cudaMemset(c->frames_d, 0, pool));   // ordered before any use: the synchronous cudaMemcpy below runs on the same (null) stream and blocks the host
    if (dalloc(c, &c->cells_d, B * c->n_cells) || dalloc(c, &c->occupied_d, B * c->n_cells) ||
        dalloc(c, &c->scoremap_d, 2 * (size_t)g.w[0] * g.h[0]) || dalloc(c, &c->ref_slots_d, B) || dalloc(c, &c->cur_slots_d, B) ||
        dalloc(c, &c->feats_d, B * F) || dalloc(c, &c->n_feats_d, B) || dalloc(c, &c->centers_d, B * 3) ||
        dalloc(c, &c->poses_in_d, B * 7) || dalloc(c, &c->poses_out_d, B * 7) || dalloc(c, &c->n_tracked_d, B) ||
        dalloc(c, &c->log_d, B * kLogCap) || dalloc(c, &c->n_log_d, B) || dalloc(c, &c->patches_d, B * P * 100) ||
        dalloc(c, &c->patch_px_d, B * P * 2) || dalloc(c, &c->patch_px_in_d, B * P * 2) || dalloc(c, &c->patch_level_d, B * P) || dalloc(c, &c->patch_slot_d, B * P) ||
        dalloc(c, &c->patch_conv_d, B * P) || dalloc(c, &c->wa_A_d, B * P * 4) || dalloc(c, &c->wa_px_d, B * P * 2) ||
        dalloc(c, &c->wa_meta_d, B * P * 3) || dalloc(c, &c->cand_d, B * P) || dalloc(c, &c->poses_ref_d, B * 7) || dalloc(c, &c->pair_reproj_d, B * P) || dalloc(c, &c->sa_ws_d, B * sparse_align_ws_doubles(prm->max_feats)))
        return bail("device buffers");
    {
        const int n = build_fast_tiles(g, nullptr, nullptr);
        std::vector<int> tiles(n);
        build_fast_tiles(g, tiles.data(), nullptr);
        c->n_fast_tiles = n;
        if (dalloc(c, &c->fast_tiles_d, (size_t)n)) return bail("fast tiles");
        CK(cudaMemcpy(c->fast_tiles_d, tiles.data(), n * sizeof(int), cudaMemcpyHostToDevice));
    }
    CK(sparse_align_init(c));
    CK(pyramid_init(c));
    CK(pose_opt_init(c));
    CK(cudaMallocHost((void**)&c->stage_pin, kStageBytes));
    CK(cudaMalloc((void**)&c->stage_dev, kStageBytes));
    CK(cudaDeviceSynchronize());   // every initialisation above (null stream) is complete before the first call uses the non-blocking streams
#undef CK
    return c;
}

void dsdtm_destroy(dsdtm_ctx* c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    for (cudaGraphExec_t g : c->batch.graph) if (g) cudaGraphExecDestroy(g);
    void* bufs[] = { c->frames_d, c->cells_d, c->occupied_d, c->scoremap_d, c->fast_tiles_d, c->ref_slots_d, c->cur_slots_d,
                     c->feats_d, c->n_feats_d, c->centers_d, c->poses_in_d, c->poses_out_d, c->n_tracked_d, c->log_d, c->n_log_d,
                     c->patches_d, c->patch_px_d, c->patch_px_in_d, c->patch_level_d, c->patch_slot_d, c->patch_conv_d, c->wa_A_d, c->wa_px_d, c->wa_meta_d, c->sa_ws_d, c->cand_d,
                     c->lm_kfs_d, c->lm_obs_d, c->lm_pts_d, c->lm_pose_d, c->lm_reproj_d, c->poses_ref_d, c->pair_reproj_d,
                     c->depth_d, c->depth_f32_d, c->lift_px_d, c->lift_initial_d, c->lift_out_d, c->clahe_src_d, c->clahe_lut_d,
                     c->po_obs_d, c->po_res_d, c->po_nobs_d, c->po_pose_in_d, c->po_pose_out_d, c->po_sum_d,
                     c->mt_kfs_d, c->mt_pts_d, c->mt_vis_d, c->mt_dist_d,
                     c->st_kfs_d, c->st_feats_d, c->st_pts_d, c->st_claim_d, c->st_vis_d, c->st_dist_d, c->st_sel_d, c->st_out_d,
                     c->trk_found_d, c->trk_match_d, c->trk_obs_d, c->trk_nobs_d, c->trk_pose_in_d, c->trk_pose_out_d, c->trk_res_d, c->trk_sum_d,
                     c->det_mask_d, c->det_buf_d, c->kf_circ_d, c->kf_ncirc_d, c->kf_max_new_d, c->kf_corner_d, c->kf_lifted_d, c->kf_nnew_d,
                     c->kf_exact_d, c->kf_depth_slot_d, c->kf_want_d, c->kf_rows_d,
                     c->sb_rec_d, c->sb_ncand_d, c->sb_local_d, c->sb_pose10_d, c->sb_range_d, c->sb_found_d,
                     c->st_found_d, c->cm_d, c->cm_push_d, c->adv_d };
    for (void* p : bufs) if (p) cudaFree(p);
    if (c->pinned) cudaFreeHost(c->pinned);
    if (c->stage_pin) cudaFreeHost(c->stage_pin);
    if (c->stage_dev) cudaFree(c->stage_dev);
    for (int i = 0; i < StageTimer::kMaxEv; ++i) { if (c->timer.ev0[i]) cudaEventDestroy(c->timer.ev0[i]); if (c->timer.ev1[i]) cudaEventDestroy(c->timer.ev1[i]); }
    for (int i = 0; i < 4; ++i) if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
    for (int i = 0; i < 8; ++i) { if (c->ev_up[i]) cudaEventDestroy(c->ev_up[i]); if (c->ev_done[i]) cudaEventDestroy(c->ev_done[i]); }
    if (c->ev_a) cudaEventDestroy(c->ev_a);
    if (c->ev_b) cudaEventDestroy(c->ev_b);
    if (c->ev_t0) cudaEventDestroy(c->ev_t0);
    if (c->ev_t1) cudaEventDestroy(c->ev_t1);
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    for (int i = 0; i < kMaxStepStreams; ++i) {
        if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]);
        if (c->step_stream[i]) cudaStreamDestroy(c->step_stream[i]);
    }
    for (int i = 0; i < 2; ++i) if (c->copy_stream[i]) cudaStreamDestroy(c->copy_stream[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* dsdtm_last_error(const dsdtm_ctx* c) { return c ? c->err.c_str() : "null context"; }

int dsdtm_sync(dsdtm_ctx* c)
{
    if (!c) return DSDTM_E_ARG;
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int dsdtm_level_info(const dsdtm_ctx* c, int level, int* w, int* h, size_t* offset)
{
    if (!c || level < 0 || level >= c->geo.levels) return DSDTM_E_ARG;
    if (w) *w = c->geo.w[level];
    if (h) *h = c->geo.h[level];
    if (offset) *offset = c->geo.off[level];
    return 0;
}

size_t dsdtm_frame_stride(const dsdtm_ctx* c) { return c ? c->geo.frame_stride : 0; }

void* dsdtm_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    return p;
}
void dsdtm_host_free(void* p) { if (p) cudaFreeHost(p); }

long long dsdtm_launch_count(const dsdtm_ctx* c) { return c ? c->launches : 0; }
long long dsdtm_graph_captures(const dsdtm_ctx* c) { return c ? c->captures : 0; }

int dsdtm_set_option(dsdtm_ctx* c, const char* key, int value)
{
    if (!c || !key) return DSDTM_E_ARG;
    if (std::strcmp(key, "sa_warps_per_pair") == 0) {
        if (value != 0 && value != 1 && value != 2 && value != 3 && value != 4 && value != 5 && value != 6 && value != 10) return fail(c, DSDTM_E_ARG, "sa_warps_per_pair must be 0, 1, 2, 3, 4, 5, 6 or 10");
        c->sa_wpp_override = value;
        drop_graphs(c);
        return 0;
    }
    if (std::strcmp(key, "sa_variant") == 0) {
        if (value != 0 && value != 1) return fail(c, DSDTM_E_ARG, "sa_variant must be 0 (shared-memory recompute) or 1 (L2 workspace)");
        c->sa_variant = value;
        drop_graphs(c);
        return 0;
    }
    if (std::strcmp(key, "step_chunks") == 0) {
        if (value < 1 || value > kMaxStepStreams) return fail(c, DSDTM_E_ARG, "step_chunks must be 1..8");
        c->step_chunks = value;
        drop_graphs(c);
        return 0;
    }
    if (std::strcmp(key, "pyramid_kernel") == 0) {
        if (value != 0 && value != 1 && value != 2) return fail(c, DSDTM_E_ARG, "pyramid_kernel must be 0 (auto: bulk-staged where eligible), 1 (tile) or 2 (register strip)");
        c->pyr_kernel = value;
        drop_graphs(c);
        return 0;
    }
    if (std::strcmp(key, "pose_opt_solo_max") == 0) {
        if (value < -1) return fail(c, DSDTM_E_ARG, "pose_opt_solo_max must be -1 (default: the SM count), 0 (always one warp per frame) or a frame count");
        c->po_solo_max = value;
        drop_graphs(c);                          // a captured dsdtm_batch_run step has its PoseOptimization kernel baked in
        return 0;
    }
    if (std::strcmp(key, "depth_slots") == 0) {
        if (value < 1 || value > 65536) return fail(c, DSDTM_E_ARG, "depth_slots must be 1..65536");
        if (c->depth_d) return fail(c, DSDTM_E_ARG, "depth_slots must be set before the depth pool is first used");
        c->depth_slots = value;
        return 0;
    }
    return fail(c, DSDTM_E_ARG, "unknown option");
}

int dsdtm_profile(dsdtm_ctx* c, int on)
{
    if (!c) return DSDTM_E_ARG;
    if (!on) stage_collect(c);
    c->profiling = on != 0;
    return 0;
}

int dsdtm_profile_get(dsdtm_ctx* c, float ms[DSDTM_STAGE_COUNT], int launches[DSDTM_STAGE_COUNT], int reset)
{
    if (!c) return DSDTM_E_ARG;
    int r = stage_collect(c);
    if (r) return r;
    for (int i = 0; i < DSDTM_STAGE_COUNT; ++i) {
        if (ms) ms[i] = c->timer.ms[i];
        if (launches) launches[i] = c->timer.launches[i];
        if (reset) { c->timer.ms[i] = 0; c->timer.launches[i] = 0; }
    }
    return 0;
}

int dsdtm_grid_dims(const dsdtm_ctx* c, int* rows, int* cols)
{
    if (!c) return DSDTM_E_ARG;
    if (rows) *rows = c->grid_rows;
    if (cols) *cols = c->grid_cols;
    return 0;
}

// ------------------------------------------------------------------------------------------------ pyramid
int dsdtm_frame_upload_pyramid(dsdtm_ctx* c, int slot, const uint8_t* img, int stride)
{
    if (!c || !img) return DSDTM_E_ARG;
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    if (stride < g.w[0]) return fail(c, DSDTM_E_ARG, "stride < width");
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)slot * g.frame_stride, g.w[0], img, stride, g.w[0], g.h[0],
                                    cudaMemcpyHostToDevice, c->stream));
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, slot, 1, c->stream));
    stage_end(c, pyramid_launches(c));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int dsdtm_frame_upload_pyramid_async(dsdtm_ctx* c, int slot, const uint8_t* img, int stride)
{
    if (!c || !img) return DSDTM_E_ARG;
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    if (stride < g.w[0]) return fail(c, DSDTM_E_ARG, "stride < width");
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)slot * g.frame_stride, g.w[0], img, stride, g.w[0], g.h[0],
                                    cudaMemcpyHostToDevice, c->stream));
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, slot, 1, c->stream));
    stage_end(c, pyramid_launches(c));
    return 0;
}

int dsdtm_frame_upload_pyramid_host(dsdtm_ctx* c, int slot, const uint8_t* img, int stride, uint8_t* levels_out)
{
    if (!c || !img) return DSDTM_E_ARG;
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    if (stride < g.w[0]) return fail(c, DSDTM_E_ARG, "stride < width");
    if (g.levels < 2) levels_out = nullptr;
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)slot * g.frame_stride, g.w[0], img, stride, g.w[0], g.h[0], cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, slot, 1, s));
    stage_end(c, pyramid_launches(c));
    const size_t tail = levels_out ? (size_t)g.off[g.levels - 1] + (size_t)g.w[g.levels - 1] * g.h[g.levels - 1] - g.off[1] : 0;
    Stager st(c, tail);
    if (levels_out)
        DSDTM_CUDA(c, cudaMemcpyAsync(st.out(levels_out, tail), c->frames_d + (size_t)slot * g.frame_stride + g.off[1], tail, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    st.finish();
    return 0;
}

int dsdtm_frames_upload_pyramid(dsdtm_ctx* c, int first_slot, int n, const uint8_t* imgs)
{
    if (!c || !imgs) return DSDTM_E_ARG;
    if (check_slot(c, first_slot, n) || check_grid_frames(c, n)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    const size_t img_bytes = (size_t)g.w[0] * g.h[0];
    // one strided copy: n rows of img_bytes into slots frame_stride apart
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)first_slot * g.frame_stride, g.frame_stride, imgs, img_bytes, img_bytes, n,
                                    cudaMemcpyHostToDevice, c->stream));
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, first_slot, n, c->stream));
    stage_end(c, pyramid_launches(c));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int dsdtm_frames_build_pyramid(dsdtm_ctx* c, int first_slot, int n)
{
    if (!c) return DSDTM_E_ARG;
    if (check_slot(c, first_slot, n) || check_grid_frames(c, n)) return DSDTM_E_ARG;
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, first_slot, n, c->stream));
    stage_end(c, pyramid_launches(c));
    return 0;
}

int dsdtm_frame_upload_level(dsdtm_ctx* c, int slot, int level, const uint8_t* img, int stride)
{
    if (!c || !img || level < 0 || level >= c->geo.levels) return c ? fail(c, DSDTM_E_ARG, "dsdtm_frame_upload_level: bad level / null image") : DSDTM_E_ARG;
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    if (stride < g.w[level]) return fail(c, DSDTM_E_ARG, "dsdtm_frame_upload_level: stride < level width");
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)slot * g.frame_stride + g.off[level], (size_t)g.w[level], img, (size_t)stride,
                                    (size_t)g.w[level], (size_t)g.h[level], cudaMemcpyHostToDevice, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int dsdtm_frame_download_level(dsdtm_ctx* c, int slot, int level, uint8_t* out)
{
    if (!c || !out || level < 0 || level >= c->geo.levels) return DSDTM_E_ARG;
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    DSDTM_CUDA(c, cudaMemcpyAsync(out, c->frames_d + (size_t)slot * g.frame_stride + g.off[level], (size_t)g.w[level] * g.h[level],
                                  cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------ FAST
int dsdtm_fast_cells_batch(dsdtm_ctx* c, int first_slot, int n, int barrier, float seed_score, const uint8_t* occupied,
                           dsdtm_corner* cells_out)
{
    if (!c || !cells_out || barrier < 1 || barrier > 254 || !(seed_score >= 0.f)) return c ? fail(c, DSDTM_E_ARG, "bad fast_cells argument") : DSDTM_E_ARG;
    if (check_slot(c, first_slot, n) || check_grid_frames(c, n)) return DSDTM_E_ARG;
    if (n > c->prm.max_batch) return fail(c, DSDTM_E_ARG, "n > max_batch");
    const size_t nc = (size_t)n * c->n_cells;
    if (occupied) DSDTM_CUDA(c, cudaMemcpyAsync(c->occupied_d, occupied, nc, cudaMemcpyHostToDevice, c->stream));
    stage_begin(c, DSDTM_STAGE_FAST);
    DSDTM_CUDA(c, launch_fast_cells(c, first_slot, n, barrier, seed_score, occupied != nullptr, c->stream));
    stage_end(c, 1);
    if (ensure_pinned(c, nc * sizeof(unsigned long long))) return DSDTM_E_NOMEM;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->pinned, c->cells_d, nc * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    decode_cells(c, reinterpret_cast<const unsigned long long*>(c->pinned), seed_score, cells_out, (int)nc);
    return 0;
}

int dsdtm_fast_cells(dsdtm_ctx* c, int slot, int barrier, float seed_score, const uint8_t* occupied, dsdtm_corner* cells_out)
{
    return dsdtm_fast_cells_batch(c, slot, 1, barrier, seed_score, occupied, cells_out);
}

int dsdtm_fast_score_map(dsdtm_ctx* c, int slot, int level, int barrier, uint8_t* score, uint8_t* nonmax)
{
    if (!c || !score || !nonmax || level < 0 || level >= c->geo.levels || barrier < 1 || barrier > 254) return DSDTM_E_ARG;
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    const size_t n = (size_t)g.w[level] * g.h[level], n0 = (size_t)g.w[0] * g.h[0];
    DSDTM_CUDA(c, cudaMemsetAsync(c->scoremap_d, 0, 2 * n0, c->stream));
    stage_begin(c, DSDTM_STAGE_FAST);
    DSDTM_CUDA(c, launch_fast_score_map(c, slot, level, barrier, c->stream));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(score, c->scoremap_d, n, cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaMemcpyAsync(nonmax, c->scoremap_d + n0, n, cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------ detect (FAST + sort + mask-circle selection)
static int check_detect(dsdtm_ctx* c, int first_slot, int n, float thr, const dsdtm_circle* circles, int circle_stride, const int* n_circles,
                        const int* max_new, int out_stride, const dsdtm_corner* out, const int* n_out)
{
    if (!out || !n_out || !max_new || n < 0 || out_stride < 0 || !(thr >= 0.f)) return fail(c, DSDTM_E_ARG, "bad detect argument");
    if (check_slot(c, first_slot, n) || check_grid_frames(c, n)) return DSDTM_E_ARG;
    if (n > c->prm.max_batch) return fail(c, DSDTM_E_ARG, "n > max_batch");
    int max_smem = 0;
    DSDTM_CUDA(c, cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
    if (!detect_select_fits(c, (size_t)max_smem))
        return fail(c, DSDTM_E_ARG, "detect: frame geometry beyond the selection bitmap (752 x 480 pixels, CellSize <= 64)");
    for (int i = 0; i < n; ++i)
        if (max_new[i] > out_stride) return fail(c, DSDTM_E_ARG, "detect: max_new > out_stride");
    if (circles) {
        if (!n_circles || circle_stride < 0) return fail(c, DSDTM_E_ARG, "detect: circles without n_circles / circle_stride");
        for (int i = 0; i < n; ++i) {
            if (n_circles[i] < 0 || n_circles[i] > circle_stride) return fail(c, DSDTM_E_ARG, "detect: n_circles out of range (circle_stride)");
            for (int q = 0; q < n_circles[i]; ++q) {
                const int r = circles[(size_t)i * circle_stride + q].radius;
                if (r < 0 || r > detect_select_max_radius()) return fail(c, DSDTM_E_ARG, "detect: circle radius out of range (0..64)");
            }
        }
    }
    return 0;
}

static int detect_submit(dsdtm_ctx* c, int first_slot, int n, float thr, bool use_occupied, const uint8_t* masks_d, const dsdtm_circle* circles_d,
                         int circle_stride, const int* n_circles_d, const int* max_new_d, dsdtm_corner* out_d, int out_stride, int* n_out_d,
                         uint8_t* exact_d)
{
    stage_begin(c, DSDTM_STAGE_FAST);
    DSDTM_CUDA(c, launch_fast_cells(c, first_slot, n, 20, thr, use_occupied, c->stream));           // ref: :81-82 barrier literal 20
    DSDTM_CUDA(c, launch_detect_select(c, n, thr, masks_d, circles_d, circle_stride, n_circles_d, max_new_d, out_d, out_stride, n_out_d,
                                       exact_d, c->stream));
    stage_end(c, 2);
    return 0;
}

int dsdtm_detect_batch(dsdtm_ctx* c, int first_slot, int n, float thr, const uint8_t* occupied, const uint8_t* masks, const dsdtm_circle* circles,
                       int circle_stride, const int* n_circles, const int* max_new, int out_stride, dsdtm_corner* out, int* n_out,
                       uint8_t* exact_path)
{
    if (!c) return DSDTM_E_ARG;
    if (int e = check_detect(c, first_slot, n, thr, circles, circle_stride, n_circles, max_new, out_stride, out, n_out)) return e;
    if (n == 0) return 0;
    auto pad = [](size_t b) { return (b + 15) & ~(size_t)15; };
    const size_t cs = circles ? (size_t)circle_stride : 0;
    // det_buf_d / pinned: max_new | n_circles | circles || n_out | exact | corners
    const size_t o_ncirc = pad(n * sizeof(int)), o_circ = o_ncirc + pad(n * sizeof(int)), in_b = o_circ + pad(n * cs * sizeof(dsdtm_circle));
    const size_t o_exact = in_b + pad(n * sizeof(int)), o_out = o_exact + pad(n), total = o_out + pad((size_t)n * out_stride * sizeof(dsdtm_corner));
    const size_t frame_px = (size_t)c->geo.w[0] * c->geo.h[0];
    if (grow(c, &c->det_buf_d, &c->det_buf_cap, total) || ensure_pinned(c, total)) return DSDTM_E_NOMEM;
    if (masks && grow(c, &c->det_mask_d, &c->det_mask_cap, n * frame_px)) return DSDTM_E_NOMEM;
    uint8_t* P = c->pinned;
    std::memcpy(P, max_new, n * sizeof(int));
    if (circles) {
        std::memcpy(P + o_ncirc, n_circles, n * sizeof(int));
        std::memcpy(P + o_circ, circles, n * cs * sizeof(dsdtm_circle));
    }
    if (occupied) DSDTM_CUDA(c, cudaMemcpyAsync(c->occupied_d, occupied, (size_t)n * c->n_cells, cudaMemcpyHostToDevice, c->stream));
    if (masks) DSDTM_CUDA(c, cudaMemcpyAsync(c->det_mask_d, masks, n * frame_px, cudaMemcpyHostToDevice, c->stream));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->det_buf_d, P, in_b, cudaMemcpyHostToDevice, c->stream));
    uint8_t* B = c->det_buf_d;
    if (detect_submit(c, first_slot, n, thr, occupied != nullptr, masks ? c->det_mask_d : nullptr,
                      circles ? reinterpret_cast<const dsdtm_circle*>(B + o_circ) : nullptr, (int)cs,
                      circles ? reinterpret_cast<const int*>(B + o_ncirc) : nullptr, reinterpret_cast<const int*>(B), reinterpret_cast<dsdtm_corner*>(B + o_out),
                      out_stride, reinterpret_cast<int*>(B + in_b), B + o_exact))
        return DSDTM_E_CUDA;
    DSDTM_CUDA(c, cudaMemcpyAsync(P + in_b, B + in_b, total - in_b, cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    std::memcpy(n_out, P + in_b, n * sizeof(int));
    if (exact_path) std::memcpy(exact_path, P + o_exact, n);
    const dsdtm_corner* R = reinterpret_cast<const dsdtm_corner*>(P + o_out);
    for (int i = 0; i < n; ++i) std::memcpy(out + (size_t)i * out_stride, R + (size_t)i * out_stride, n_out[i] * sizeof(dsdtm_corner));
    return 0;
}

int dsdtm_detect(dsdtm_ctx* c, int slot, float thr, const uint8_t* occupied, const uint8_t* mask, const dsdtm_circle* circles, int n_circles,
                 int max_new, dsdtm_corner* out, int* n_out, uint8_t* exact_path)
{
    if (!c) return DSDTM_E_ARG;
    if (n_circles < 0 || (n_circles > 0 && !circles)) return fail(c, DSDTM_E_ARG, "detect: n_circles < 0 or circles NULL");
    const int nc = circles ? n_circles : 0, stride = std::max(max_new, 0);
    if (int e = check_detect(c, slot, 1, thr, circles, nc, &nc, &max_new, stride, out, n_out)) return e;
    const size_t frame_px = (size_t)c->geo.w[0] * c->geo.h[0];
    const size_t in_b = (occupied ? c->n_cells : 0) + (mask ? frame_px : 0) + 2 * sizeof(int) + nc * sizeof(dsdtm_circle);
    const size_t out_b = sizeof(int) + 1 + (size_t)stride * sizeof(dsdtm_corner);
    Arena ar(c, in_b, out_b, 5, 3);
    if (!ar.active)
        return dsdtm_detect_batch(c, slot, 1, thr, occupied, mask, circles, nc, &nc, &max_new, stride, out, n_out, exact_path);
    uint8_t* occ_d = occupied ? ar.in(occupied, c->n_cells) : nullptr;
    const uint8_t* mask_d = mask ? ar.in(mask, frame_px) : nullptr;
    const int* max_new_d = ar.in(&max_new, 1);
    const int* nc_d = ar.in(&nc, 1);
    const dsdtm_circle* circ_d = nc ? ar.in(circles, nc) : nullptr;
    uint8_t exact = 0;
    int* n_out_d = ar.out(n_out, 1);
    uint8_t* exact_d = ar.out(&exact, 1);
    dsdtm_corner* out_d = ar.out(static_cast<dsdtm_corner*>(nullptr), std::max(stride, 1));
    DSDTM_CUDA(c, ar.upload(c->stream));
    {
        PtrSwap<uint8_t> sw(c->occupied_d, occ_d ? occ_d : c->occupied_d);
        if (detect_submit(c, slot, 1, thr, occ_d != nullptr, mask_d, circ_d, nc, circ_d ? nc_d : nullptr, max_new_d, out_d, stride, n_out_d, exact_d))
            return DSDTM_E_CUDA;
    }
    DSDTM_CUDA(c, ar.download(c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    ar.finish();
    std::memcpy(out, ar.host_view(out_d), *n_out * sizeof(dsdtm_corner));
    if (exact_path) *exact_path = exact;
    return 0;
}

// ------------------------------------------------------------------------------------------------ sparse align
static int stage_pairs(dsdtm_ctx* c, int n_pairs, const int* ref_slots, const int* cur_slots, const dsdtm_ref_feat* feats,
                       int feat_stride, const int* n_feats, const double* ref_centers, const double* poses_in, cudaStream_t s,
                       int pair0 = 0, Stager* st = nullptr)
{
    auto src = [&](const void* p, size_t bytes) { return st ? st->in(p, bytes) : p; };
    DSDTM_CUDA(c, cudaMemcpyAsync(c->ref_slots_d + pair0, src(ref_slots + pair0, n_pairs * sizeof(int)), n_pairs * sizeof(int), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->cur_slots_d + pair0, src(cur_slots + pair0, n_pairs * sizeof(int)), n_pairs * sizeof(int), cudaMemcpyHostToDevice, s));
    const size_t fb = (size_t)n_pairs * feat_stride * sizeof(dsdtm_ref_feat);
    DSDTM_CUDA(c, cudaMemcpyAsync(c->feats_d + (size_t)pair0 * feat_stride, src(feats + (size_t)pair0 * feat_stride, fb), fb, cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->n_feats_d + pair0, src(n_feats + pair0, n_pairs * sizeof(int)), n_pairs * sizeof(int), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->centers_d + 3 * (size_t)pair0, src(ref_centers + 3 * (size_t)pair0, (size_t)n_pairs * 3 * sizeof(double)),
                                  (size_t)n_pairs * 3 * sizeof(double), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->poses_in_d + 7 * (size_t)pair0, src(poses_in + 7 * (size_t)pair0, (size_t)n_pairs * 7 * sizeof(double)),
                                  (size_t)n_pairs * 7 * sizeof(double), cudaMemcpyHostToDevice, s));
    return 0;
}

static int check_pairs(dsdtm_ctx* c, int n_pairs, const int* ref_slots, const int* cur_slots, int feat_stride, const int* n_feats,
                       int max_level, int min_level, int max_iters)
{
    if (n_pairs < 1 || n_pairs > c->prm.max_batch) return fail(c, DSDTM_E_ARG, "n_pairs out of range (max_batch)");
    if (feat_stride < 1 || feat_stride > c->prm.max_feats) return fail(c, DSDTM_E_ARG, "feat_stride > max_feats");
    if (max_level < 1 || max_level > c->geo.levels || min_level < 0 || min_level >= max_level || max_iters < 0)
        return fail(c, DSDTM_E_ARG, "bad level range / iterations");
    for (int i = 0; i < n_pairs; ++i) {
        if (ref_slots[i] < 0 || ref_slots[i] >= c->prm.max_frames || cur_slots[i] < 0 || cur_slots[i] >= c->prm.max_frames)
            return fail(c, DSDTM_E_ARG, "pair slot out of range");
        if (n_feats[i] < 0 || n_feats[i] > feat_stride) return fail(c, DSDTM_E_ARG, "n_feats > feat_stride");
    }
    return 0;
}

int dsdtm_sparse_align_batch(dsdtm_ctx* c, int n_pairs, const int* ref_slots, const int* cur_slots, const dsdtm_ref_feat* feats,
                             int feat_stride, const int* n_feats, const double* ref_centers, const double* poses_in, int max_level,
                             int min_level, int max_iters, double* poses_out, int* n_tracked, dsdtm_iter_log* log,
                             int log_cap_per_pair, int* n_log)
{
    if (!c || !ref_slots || !cur_slots || !feats || !n_feats || !ref_centers || !poses_in || !poses_out || !n_tracked) return DSDTM_E_ARG;
    if (check_pairs(c, n_pairs, ref_slots, cur_slots, feat_stride, n_feats, max_level, min_level, max_iters)) return DSDTM_E_ARG;
    c->batch.staged = false;
    const bool want_log = log != nullptr && log_cap_per_pair > 0;
    const size_t log_bytes = want_log ? (size_t)n_pairs * (kLogCap * sizeof(dsdtm_iter_log) + sizeof(int)) : 0;
    {
        const size_t nfe = (size_t)n_pairs * feat_stride;
        Arena ar(c, (size_t)n_pairs * (3 * sizeof(int) + 10 * sizeof(double)) + nfe * sizeof(dsdtm_ref_feat),
                 (size_t)n_pairs * (7 * sizeof(double) + 2 * sizeof(int)) + (size_t)n_pairs * kLogCap * sizeof(dsdtm_iter_log), 6, 4);
        if (ar.active) {
            cudaStream_t s = c->stream;
            PtrSwap<int> p0(c->ref_slots_d, ar.in(ref_slots, n_pairs)), p1(c->cur_slots_d, ar.in(cur_slots, n_pairs)), p2(c->n_feats_d, ar.in(n_feats, n_pairs));
            PtrSwap<double> p3(c->centers_d, ar.in(ref_centers, (size_t)n_pairs * 3)), p4(c->poses_in_d, ar.in(poses_in, (size_t)n_pairs * 7));
            PtrSwap<dsdtm_ref_feat> p5(c->feats_d, ar.in(feats, nfe));
            PtrSwap<double> q0(c->poses_out_d, ar.out(poses_out, (size_t)n_pairs * 7));
            PtrSwap<int> q1(c->n_tracked_d, ar.out(n_tracked, n_pairs)), q2(c->n_log_d, ar.out((int*)nullptr, n_pairs));
            // the log travels back only when it is wanted: it is the last range, download() stops before it otherwise
            const size_t end_no_log = ar.out_end;
            PtrSwap<dsdtm_iter_log> q3(c->log_d, ar.out((dsdtm_iter_log*)nullptr, (size_t)n_pairs * kLogCap));
            if (!want_log) ar.out_end = end_no_log;
            DSDTM_CUDA(c, ar.upload(s));
            stage_begin(c, DSDTM_STAGE_SPARSE_ALIGN);
            DSDTM_CUDA(c, launch_sparse_align(c, n_pairs, feat_stride, max_level, min_level, max_iters, want_log, s));
            stage_end(c, 1);
            DSDTM_CUDA(c, ar.download(s));
            DSDTM_CUDA(c, cudaStreamSynchronize(s));
            ar.finish();
            const int* hn = ar.host_view(c->n_log_d);
            const dsdtm_iter_log* hl = ar.host_view(c->log_d);
            for (int i = 0; i < n_pairs; ++i) {
                if (want_log) {
                    const int n = std::min(std::min(hn[i], kLogCap), log_cap_per_pair);
                    std::memcpy(log + (size_t)i * log_cap_per_pair, hl + (size_t)i * kLogCap, n * sizeof(dsdtm_iter_log));
                }
                if (n_log) n_log[i] = want_log ? hn[i] : 0;
            }
            return 0;
        }
    }
    Stager st(c, (size_t)n_pairs * (3 * sizeof(int) + 10 * sizeof(double) + (size_t)feat_stride * sizeof(dsdtm_ref_feat)) +
                 (size_t)n_pairs * (7 * sizeof(double) + sizeof(int)) + log_bytes);
    if (stage_pairs(c, n_pairs, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_in, c->stream, 0, &st)) return DSDTM_E_CUDA;
    stage_begin(c, DSDTM_STAGE_SPARSE_ALIGN);
    DSDTM_CUDA(c, launch_sparse_align(c, n_pairs, feat_stride, max_level, min_level, max_iters, want_log, c->stream));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(poses_out, (size_t)n_pairs * 7 * sizeof(double)), c->poses_out_d, (size_t)n_pairs * 7 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(n_tracked, n_pairs * sizeof(int)), c->n_tracked_d, n_pairs * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    if (want_log) {
        dsdtm_iter_log* hl;
        int* hn;
        if (st.active) {
            hl = reinterpret_cast<dsdtm_iter_log*>(st.carve((size_t)n_pairs * kLogCap * sizeof(dsdtm_iter_log)));
            hn = reinterpret_cast<int*>(st.carve((size_t)n_pairs * sizeof(int)));
        } else {
            if (ensure_pinned(c, log_bytes)) return DSDTM_E_NOMEM;
            hl = reinterpret_cast<dsdtm_iter_log*>(c->pinned);
            hn = reinterpret_cast<int*>(c->pinned + (size_t)n_pairs * kLogCap * sizeof(dsdtm_iter_log));
        }
        DSDTM_CUDA(c, cudaMemcpyAsync(hn, c->n_log_d, n_pairs * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        DSDTM_CUDA(c, cudaMemcpyAsync(hl, c->log_d, (size_t)n_pairs * kLogCap * sizeof(dsdtm_iter_log), cudaMemcpyDeviceToHost, c->stream));
        DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
        st.finish();
        for (int i = 0; i < n_pairs; ++i) {
            const int n = std::min(std::min(hn[i], kLogCap), log_cap_per_pair);
            std::memcpy(log + (size_t)i * log_cap_per_pair, hl + (size_t)i * kLogCap, n * sizeof(dsdtm_iter_log));
            if (n_log) n_log[i] = hn[i];
        }
    } else {
        DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
        st.finish();
        if (n_log) for (int i = 0; i < n_pairs; ++i) n_log[i] = 0;
    }
    return 0;
}

int dsdtm_sparse_align(dsdtm_ctx* c, int ref_slot, int cur_slot, const dsdtm_ref_feat* feats, int n_feats, const double ref_center[3],
                       const double pose_in[7], int max_level, int min_level, int max_iters, double pose_out[7], int* n_tracked,
                       dsdtm_iter_log* log, int log_cap, int* n_log)
{
    if (!c) return DSDTM_E_ARG;
    if (n_feats < 1 || n_feats > c->prm.max_feats) return fail(c, DSDTM_E_ARG, "n_feats out of range (max_feats)");
    return dsdtm_sparse_align_batch(c, 1, &ref_slot, &cur_slot, feats, n_feats, &n_feats, ref_center, pose_in, max_level, min_level,
                                    max_iters, pose_out, n_tracked, log, log_cap, n_log);
}

// ------------------------------------------------------------------------------------------------ align2d / warp
int dsdtm_align2d_batch(dsdtm_ctx* c, int cur_slot, const int* level, const uint8_t* patch10, double* px_io, int n, int max_iters,
                        uint8_t* converged)
{
    if (!c || !level || !patch10 || !px_io || !converged || n < 0 || max_iters < 0) return DSDTM_E_ARG;
    if (check_slot(c, cur_slot)) return DSDTM_E_ARG;
    if (n == 0) return 0;
    const size_t cap = (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1);
    if ((size_t)n > cap) return fail(c, DSDTM_E_ARG, "n > max_batch * max_patches");
    for (int i = 0; i < n; ++i) if (level[i] >= c->geo.levels) return fail(c, DSDTM_E_ARG, "patch level out of range");
    c->batch.staged = false;
    {
        Arena ar(c, (size_t)n * (2 * sizeof(int) + 100 + 2 * sizeof(double)), (size_t)n * (2 * sizeof(double) + 1), 4, 2);
        if (ar.active) {
            cudaStream_t s = c->stream;
            int* slots_h;
            PtrSwap<int> p0(c->patch_slot_d, ar.in_fill(n, &slots_h)), p1(c->patch_level_d, ar.in(level, n));
            for (int i = 0; i < n; ++i) slots_h[i] = cur_slot;
            PtrSwap<uint8_t> p2(c->patches_d, ar.in(patch10, (size_t)n * 100));
            PtrSwap<double> p3(c->patch_px_in_d, ar.in(px_io, (size_t)n * 2)), q0(c->patch_px_d, ar.out(px_io, (size_t)n * 2));
            PtrSwap<uint8_t> q1(c->patch_conv_d, ar.out(converged, n));
            DSDTM_CUDA(c, ar.upload(s));
            stage_begin(c, DSDTM_STAGE_ALIGN2D);
            DSDTM_CUDA(c, launch_align2d(c, n, max_iters, s));
            stage_end(c, 1);
            DSDTM_CUDA(c, ar.download(s));
            DSDTM_CUDA(c, cudaStreamSynchronize(s));
            ar.finish();
            return 0;
        }
    }
    if (ensure_pinned(c, (size_t)n * sizeof(int))) return DSDTM_E_NOMEM;
    int* slots = reinterpret_cast<int*>(c->pinned);
    for (int i = 0; i < n; ++i) slots[i] = cur_slot;
    cudaStream_t s = c->stream;
    Stager st(c, (size_t)n * (sizeof(int) + 100 + 4 * sizeof(double) + 1));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patch_slot_d, slots, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patch_level_d, st.in(level, (size_t)n * sizeof(int)), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patches_d, st.in(patch10, (size_t)n * 100), (size_t)n * 100, cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patch_px_in_d, st.in(px_io, (size_t)n * 2 * sizeof(double)), (size_t)n * 2 * sizeof(double), cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_ALIGN2D);
    DSDTM_CUDA(c, launch_align2d(c, n, max_iters, s));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(px_io, (size_t)n * 2 * sizeof(double)), c->patch_px_d, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(converged, (size_t)n), c->patch_conv_d, (size_t)n, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    st.finish();
    return 0;
}

int dsdtm_warp_affine_batch(dsdtm_ctx* c, const int* ref_slot, const double* A, const float* ref_px, const int* ref_level,
                            const int* search_level, int n, uint8_t* patch10_out)
{
    if (!c || !ref_slot || !A || !ref_px || !ref_level || !search_level || !patch10_out || n < 0) return DSDTM_E_ARG;
    if (n == 0) return 0;
    const size_t cap = (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1);
    if ((size_t)n > cap) return fail(c, DSDTM_E_ARG, "n > max_batch * max_patches");
    if (ensure_pinned(c, (size_t)n * 3 * sizeof(int))) return DSDTM_E_NOMEM;
    int* meta = reinterpret_cast<int*>(c->pinned);
    for (int i = 0; i < n; ++i) {
        if (ref_slot[i] < 0 || ref_slot[i] >= c->prm.max_frames || ref_level[i] < 0 || ref_level[i] >= c->geo.levels ||
            search_level[i] < 0 || search_level[i] > 30)
            return fail(c, DSDTM_E_ARG, "warp_affine: slot / level out of range");
        meta[3 * i] = ref_slot[i]; meta[3 * i + 1] = ref_level[i]; meta[3 * i + 2] = search_level[i];
    }
    c->batch.staged = false;
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->wa_meta_d, meta, (size_t)n * 3 * sizeof(int), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->wa_A_d, A, (size_t)n * 4 * sizeof(double), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->wa_px_d, ref_px, (size_t)n * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
    DSDTM_CUDA(c, launch_warp_affine(c, n, c->patches_d, s));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(patch10_out, c->patches_d, (size_t)n * 100, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

int dsdtm_feature_align_batch(dsdtm_ctx* c, int cur_slot, const dsdtm_candidate* cands, int n, int max_search_level, int max_iters,
                              double* px_out, int* level_out, uint8_t* converged, double* A_out)
{
    if (!c || !cands || !px_out || !level_out || !converged || n < 0 || max_iters < 0 || max_search_level < 0) return DSDTM_E_ARG;
    if (check_slot(c, cur_slot)) return DSDTM_E_ARG;
    if (n == 0) return 0;
    const size_t cap = (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1);
    if ((size_t)n > cap) return fail(c, DSDTM_E_ARG, "n > max_batch * max_patches");
    if (max_search_level >= c->geo.levels) return fail(c, DSDTM_E_ARG, "max_search_level >= levels");
    for (int i = 0; i < n; ++i)
        if (cands[i].ref_slot < 0 || cands[i].ref_slot >= c->prm.max_frames || cands[i].ref_level < 0 || cands[i].ref_level >= c->geo.levels)
            return fail(c, DSDTM_E_ARG, "candidate: slot / level out of range");
    c->batch.staged = false;
    cudaStream_t s = c->stream;
    Stager st(c, (size_t)n * (sizeof(dsdtm_candidate) + 2 * sizeof(double) + sizeof(int) + 1 + (A_out ? 4 * sizeof(double) : 0)));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->cand_d, st.in(cands, (size_t)n * sizeof(dsdtm_candidate)), (size_t)n * sizeof(dsdtm_candidate), cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_CAND_PREP);
    DSDTM_CUDA(c, launch_candidate_prep(c, n, cur_slot, max_search_level, s));
    stage_end(c, 1);
    stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
    DSDTM_CUDA(c, launch_warp_affine(c, n, c->patches_d, s));
    stage_end(c, 1);
    stage_begin(c, DSDTM_STAGE_ALIGN2D);
    DSDTM_CUDA(c, launch_align2d(c, n, max_iters, s));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(px_out, (size_t)n * 2 * sizeof(double)), c->patch_px_d, (size_t)n * 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(level_out, (size_t)n * sizeof(int)), c->patch_level_d, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(converged, (size_t)n), c->patch_conv_d, (size_t)n, cudaMemcpyDeviceToHost, s));
    if (A_out) DSDTM_CUDA(c, cudaMemcpyAsync(st.out(A_out, (size_t)n * 4 * sizeof(double)), c->wa_A_d, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    st.finish();
    for (int i = 0; i < n; ++i) {                                   // ref: :154 tPt = tCurPx * (1 << tBestLevel) (exact)
        const double sc = (double)(1 << level_out[i]);
        px_out[2 * i] *= sc; px_out[2 * i + 1] *= sc;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------ (f-1) local map
int dsdtm_local_map_align_batch(dsdtm_ctx* c, int cur_slot, const double pose_cur_c2w[7], const double cur_center[3],
                                const dsdtm_kf_view* kfs, int n_kfs, const dsdtm_obs* obs, int n_obs, const dsdtm_map_point* pts,
                                int n_pts, int max_search_level, int max_iters, dsdtm_reproj* out)
{
    if (!c || !pose_cur_c2w || !cur_center || n_kfs < 0 || n_obs < 0 || n_pts < 0 || max_iters < 0 || max_search_level < 0) return DSDTM_E_ARG;
    if ((n_kfs && !kfs) || (n_obs && !obs) || (n_pts && (!pts || !out))) return fail(c, DSDTM_E_ARG, "null table");
    if (check_slot(c, cur_slot)) return DSDTM_E_ARG;
    if (n_pts == 0) return 0;
    const size_t cap = (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1);
    if ((size_t)n_pts > cap) return fail(c, DSDTM_E_ARG, "n_pts > max_batch * max_patches");
    if (max_search_level >= c->geo.levels) return fail(c, DSDTM_E_ARG, "max_search_level >= levels");
    for (int k = 0; k < n_kfs; ++k)
        if (kfs[k].slot < 0 || kfs[k].slot >= c->prm.max_frames) return fail(c, DSDTM_E_ARG, "keyframe: slot out of range");
    for (int j = 0; j < n_obs; ++j)
        if (obs[j].kf < 0 || obs[j].kf >= n_kfs || obs[j].level < 0 || obs[j].level >= c->geo.levels)
            return fail(c, DSDTM_E_ARG, "observation: keyframe index / level out of range");
    for (int i = 0; i < n_pts; ++i)
        if (pts[i].obs_count < 0 || pts[i].obs_begin < 0 || (long long)pts[i].obs_begin + pts[i].obs_count > n_obs)
            return fail(c, DSDTM_E_ARG, "map point: observation range out of bounds");
    c->batch.staged = false;
    {
        const size_t kcap0 = c->lm_kfs_cap, pcap0 = c->lm_pts_cap;
        if (grow(c, &c->lm_kfs_d, &c->lm_kfs_cap, (size_t)n_kfs) || grow(c, &c->lm_obs_d, &c->lm_obs_cap, (size_t)n_obs) ||
            grow(c, &c->lm_pts_d, &c->lm_pts_cap, (size_t)n_pts))
            return DSDTM_E_NOMEM;
        if (c->lm_kfs_cap != kcap0) { size_t z = 0; if (grow(c, &c->lm_pose_d, &z, c->lm_kfs_cap * 7)) return DSDTM_E_NOMEM; }
        if (c->lm_pts_cap != pcap0) { size_t z = 0; if (grow(c, &c->lm_reproj_d, &z, c->lm_pts_cap)) return DSDTM_E_NOMEM; }
    }
    cudaStream_t s = c->stream;
    const size_t kb = (size_t)n_kfs * sizeof(dsdtm_kf_view), ob = (size_t)n_obs * sizeof(dsdtm_obs), pb = (size_t)n_pts * sizeof(dsdtm_map_point);
    const size_t rb = (size_t)n_pts * sizeof(dsdtm_reproj);
    auto chain = [&]() -> int {
        stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
        DSDTM_CUDA(c, launch_local_map(c, pose_cur_c2w, cur_center, n_kfs, n_pts, s));
        stage_end(c, 2);
        stage_begin(c, DSDTM_STAGE_CAND_PREP);
        DSDTM_CUDA(c, launch_candidate_prep(c, n_pts, cur_slot, max_search_level, s));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
        DSDTM_CUDA(c, launch_warp_affine(c, n_pts, c->patches_d, s));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_ALIGN2D);
        DSDTM_CUDA(c, launch_align2d(c, n_pts, max_iters, s));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
        DSDTM_CUDA(c, launch_local_map_finalize(c, n_pts, s));
        stage_end(c, 1);
        return 0;
    };
    Arena ar(c, kb + ob + pb, rb, 3, 1);
    if (ar.active) {                                                // one copy in, six small kernels, one copy out
        dsdtm_kf_view kf_dummy{};
        dsdtm_obs obs_dummy{};
        PtrSwap<dsdtm_kf_view> p0(c->lm_kfs_d, ar.in(n_kfs ? kfs : &kf_dummy, n_kfs ? (size_t)n_kfs : 1));
        PtrSwap<dsdtm_obs> p1(c->lm_obs_d, ar.in(n_obs ? obs : &obs_dummy, n_obs ? (size_t)n_obs : 1));
        PtrSwap<dsdtm_map_point> p2(c->lm_pts_d, ar.in(pts, (size_t)n_pts));
        PtrSwap<dsdtm_reproj> q0(c->lm_reproj_d, ar.out(out, (size_t)n_pts));
        DSDTM_CUDA(c, ar.upload(s));
        if (chain()) return DSDTM_E_CUDA;
        DSDTM_CUDA(c, ar.download(s));
        DSDTM_CUDA(c, cudaStreamSynchronize(s));
        ar.finish();
        return 0;
    }
    if (n_kfs) DSDTM_CUDA(c, cudaMemcpyAsync(c->lm_kfs_d, kfs, kb, cudaMemcpyHostToDevice, s));
    if (n_obs) DSDTM_CUDA(c, cudaMemcpyAsync(c->lm_obs_d, obs, ob, cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->lm_pts_d, pts, pb, cudaMemcpyHostToDevice, s));
    if (chain()) return DSDTM_E_CUDA;
    DSDTM_CUDA(c, cudaMemcpyAsync(out, c->lm_reproj_d, rb, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------------------------------------ one call per frame
int dsdtm_track_frame(dsdtm_ctx* c, const dsdtm_track_in* in, dsdtm_track_out* out, dsdtm_reproj* reproj)
{
    if (!c || !in || !out || !in->img || !in->feats) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    const int nf = in->n_feats, n_kfs = in->n_kfs, n_obs = in->n_obs, n_pts = in->n_pts;
    if (nf < 1 || nf > c->prm.max_feats) return fail(c, DSDTM_E_ARG, "n_feats out of range (max_feats)");
    if (check_pairs(c, 1, &in->ref_slot, &in->cur_slot, nf, &nf, in->max_level, in->min_level, in->max_iters)) return DSDTM_E_ARG;
    if (in->stride < g.w[0]) return fail(c, DSDTM_E_ARG, "stride < width");
    if (n_kfs < 0 || n_obs < 0 || n_pts < 0 || in->align_iters < 0 || in->max_search_level < 0 || in->max_search_level >= g.levels)
        return fail(c, DSDTM_E_ARG, "bad local-map arguments");
    if ((n_kfs && !in->kfs) || (n_obs && !in->obs) || (n_pts && (!in->pts || !reproj))) return fail(c, DSDTM_E_ARG, "null table");
    if ((size_t)n_pts > (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1)) return fail(c, DSDTM_E_ARG, "n_pts > max_batch * max_patches");
    for (int k = 0; k < n_kfs; ++k)
        if (in->kfs[k].slot < 0 || in->kfs[k].slot >= c->prm.max_frames) return fail(c, DSDTM_E_ARG, "keyframe: slot out of range");
    for (int j = 0; j < n_obs; ++j)
        if (in->obs[j].kf < 0 || in->obs[j].kf >= n_kfs || in->obs[j].level < 0 || in->obs[j].level >= g.levels)
            return fail(c, DSDTM_E_ARG, "observation: keyframe index / level out of range");
    for (int i = 0; i < n_pts; ++i)
        if (in->pts[i].obs_count < 0 || in->pts[i].obs_begin < 0 || (long long)in->pts[i].obs_begin + in->pts[i].obs_count > n_obs)
            return fail(c, DSDTM_E_ARG, "map point: observation range out of bounds");
    const size_t kb = (size_t)std::max(n_kfs, 1) * sizeof(dsdtm_kf_view), ob = (size_t)std::max(n_obs, 1) * sizeof(dsdtm_obs);
    const size_t pb = (size_t)std::max(n_pts, 1) * sizeof(dsdtm_map_point), rb = (size_t)std::max(n_pts, 1) * sizeof(dsdtm_reproj);
    Arena ar(c, 3 * sizeof(int) + 10 * sizeof(double) + (size_t)nf * sizeof(dsdtm_ref_feat) + kb + ob + pb,
             (7 + 10) * sizeof(double) + 2 * sizeof(int) + rb, 9, 5);
    if (!ar.active) return fail(c, DSDTM_E_ARG, "dsdtm_track_frame: inputs exceed the 1 MB staging arena (use the separate calls)");
    {   // the per-keyframe pose scratch follows the capacity of the keyframe table (before any pointer is swapped)
        const size_t kcap0 = c->lm_kfs_cap;
        if (grow(c, &c->lm_kfs_d, &c->lm_kfs_cap, (size_t)std::max(n_kfs, 1))) return DSDTM_E_NOMEM;
        if (c->lm_kfs_cap != kcap0) { size_t z = 0; if (grow(c, &c->lm_pose_d, &z, c->lm_kfs_cap * 7)) return DSDTM_E_NOMEM; }
    }
    c->batch.staged = false;
    cudaStream_t s = c->stream;
    dsdtm_kf_view kf_dummy{};
    dsdtm_obs obs_dummy{};
    dsdtm_map_point pt_dummy{};
    PtrSwap<int> p0(c->ref_slots_d, ar.in(&in->ref_slot, 1)), p1(c->cur_slots_d, ar.in(&in->cur_slot, 1)), p2(c->n_feats_d, ar.in(&nf, 1));
    PtrSwap<double> p3(c->centers_d, ar.in(in->ref_center, 3)), p4(c->poses_in_d, ar.in(in->pose_c2r_in, 7));
    PtrSwap<dsdtm_ref_feat> p5(c->feats_d, ar.in(in->feats, (size_t)nf));
    PtrSwap<dsdtm_kf_view> p6(c->lm_kfs_d, ar.in(n_kfs ? in->kfs : &kf_dummy, (size_t)std::max(n_kfs, 1)));
    PtrSwap<dsdtm_obs> p7(c->lm_obs_d, ar.in(n_obs ? in->obs : &obs_dummy, (size_t)std::max(n_obs, 1)));
    PtrSwap<dsdtm_map_point> p8(c->lm_pts_d, ar.in(n_pts ? in->pts : &pt_dummy, (size_t)std::max(n_pts, 1)));
    double* pose_c2r_d = ar.out(out->pose_c2r, 7);
    double* pose10_d = ar.out((double*)nullptr, 10);
    PtrSwap<double> q0(c->poses_out_d, pose_c2r_d);
    PtrSwap<int> q1(c->n_tracked_d, ar.out(&out->n_tracked, 1)), q2(c->n_log_d, ar.out((int*)nullptr, 1));
    PtrSwap<dsdtm_reproj> q3(c->lm_reproj_d, ar.out(n_pts ? reproj : (dsdtm_reproj*)nullptr, (size_t)std::max(n_pts, 1)));
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)in->cur_slot * g.frame_stride, g.w[0], in->img, in->stride, g.w[0], g.h[0], cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, ar.upload(s));
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, in->cur_slot, 1, s));
    stage_end(c, pyramid_launches(c));
    stage_begin(c, DSDTM_STAGE_SPARSE_ALIGN);
    DSDTM_CUDA(c, launch_sparse_align(c, 1, nf, in->max_level, in->min_level, in->max_iters, false, s));
    stage_end(c, 1);
    stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
    DSDTM_CUDA(c, launch_compose_pose(c, pose_c2r_d, in->pose_ref_c2w, pose10_d, s));
    stage_end(c, 1);
    if (n_pts > 0) {
        stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
        DSDTM_CUDA(c, launch_local_map(c, nullptr, nullptr, n_kfs, n_pts, s, pose10_d));
        stage_end(c, 2);
        stage_begin(c, DSDTM_STAGE_CAND_PREP);
        DSDTM_CUDA(c, launch_candidate_prep(c, n_pts, in->cur_slot, in->max_search_level, s));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
        DSDTM_CUDA(c, launch_warp_affine(c, n_pts, c->patches_d, s));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_ALIGN2D);
        DSDTM_CUDA(c, launch_align2d(c, n_pts, in->align_iters, s));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
        DSDTM_CUDA(c, launch_local_map_finalize(c, n_pts, s));
        stage_end(c, 1);
    }
    DSDTM_CUDA(c, ar.download(s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    ar.finish();
    const double* p10 = ar.host_view(pose10_d);
    for (int k = 0; k < 7; ++k) out->pose_cur_c2w[k] = p10[k];
    for (int k = 0; k < 3; ++k) out->cur_center[k] = p10[7 + k];
    out->reserved = 0;
    return 0;
}

// ------------------------------------------------------------------------------------------------ (f-3 / f-4) ingest
static int ensure_depth_pool(dsdtm_ctx* c)
{
    if (c->depth_d) return 0;
    const size_t px = (size_t)c->cam.width * c->cam.height;
    if (dalloc(c, &c->depth_d, px * c->depth_slots)) return DSDTM_E_NOMEM;
    // on the context's stream: it is a non-blocking stream, so a memset on the null stream is NOT ordered with the uploads that
    // follow and could land after the first one (seen once as a zeroed slot 0 in test_depth_convert_bit_exact)
    cudaError_t e = cudaMemsetAsync(c->depth_d, 0, px * c->depth_slots * sizeof(uint16_t), c->stream);
    if (e != cudaSuccess) return fail(c, DSDTM_E_CUDA, "cudaMemsetAsync(depth pool)", e);
    return 0;
}

int dsdtm_depth_upload(dsdtm_ctx* c, int depth_slot, const uint16_t* depth, int stride_bytes)
{
    if (!c || !depth) return DSDTM_E_ARG;
    if (depth_slot < 0 || depth_slot >= c->depth_slots) return fail(c, DSDTM_E_ARG, "depth slot out of range (option depth_slots)");
    const int w = c->cam.width, h = c->cam.height;
    if (stride_bytes == 0) stride_bytes = 2 * w;
    if (stride_bytes < 2 * w) return fail(c, DSDTM_E_ARG, "depth stride < 2 * width");
    if (ensure_depth_pool(c)) return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpy2DAsync(c->depth_d + (size_t)depth_slot * w * h, 2 * (size_t)w, depth, (size_t)stride_bytes, 2 * (size_t)w, h,
                                    cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

int dsdtm_depth_convert_f32(dsdtm_ctx* c, int first_depth_slot, int n, float depth_scale, float* out)
{
    if (!c || n < 0) return DSDTM_E_ARG;
    if (first_depth_slot < 0 || first_depth_slot + n > c->depth_slots) return fail(c, DSDTM_E_ARG, "depth slot range out of bounds (option depth_slots)");
    if (!(depth_scale > 0.f)) return fail(c, DSDTM_E_ARG, "depth_scale must be > 0");
    if (n == 0) return 0;
    if (ensure_depth_pool(c)) return DSDTM_E_NOMEM;
    const size_t px = (size_t)c->cam.width * c->cam.height;
    if (!c->depth_f32_d && dalloc(c, &c->depth_f32_d, px * c->depth_slots)) return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    stage_begin(c, DSDTM_STAGE_INGEST);
    DSDTM_CUDA(c, launch_depth_convert(c, first_depth_slot, n, depth_scale, s));
    stage_end(c, 1);
    if (out) DSDTM_CUDA(c, cudaMemcpyAsync(out, c->depth_f32_d + (size_t)first_depth_slot * px, px * n * sizeof(float), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

int dsdtm_keyframe_lift(dsdtm_ctx* c, int depth_slot, const double pose_c2w[7], const float dist[5], float depth_scale,
                        const float* px_in, const uint8_t* initial, int n, dsdtm_lifted* out)
{
    if (!c || !pose_c2w || !dist || n < 0 || (n && (!px_in || !out))) return DSDTM_E_ARG;
    if (depth_slot >= c->depth_slots) return fail(c, DSDTM_E_ARG, "depth slot out of range (option depth_slots)");
    if (depth_slot >= 0 && !(depth_scale > 0.f)) return fail(c, DSDTM_E_ARG, "depth_scale must be > 0");
    if (n == 0) return 0;
    if (depth_slot >= 0 && ensure_depth_pool(c)) return DSDTM_E_NOMEM;
    if ((size_t)n > c->lift_cap) {
        size_t z0 = 0, z1 = 0, z2 = 0;
        const size_t want = std::max<size_t>((size_t)n, 512);
        if (c->lift_px_d) { cudaFree(c->lift_px_d); c->lift_px_d = nullptr; }
        if (c->lift_initial_d) { cudaFree(c->lift_initial_d); c->lift_initial_d = nullptr; }
        if (c->lift_out_d) { cudaFree(c->lift_out_d); c->lift_out_d = nullptr; }
        c->lift_cap = 0;
        if (grow(c, &c->lift_px_d, &z0, 2 * want) || grow(c, &c->lift_initial_d, &z1, want) || grow(c, &c->lift_out_d, &z2, want)) return DSDTM_E_NOMEM;
        c->lift_cap = want;
    }
    cudaStream_t s = c->stream;
    Stager st(c, (size_t)n * (2 * sizeof(float) + 1 + sizeof(dsdtm_lifted)));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->lift_px_d, st.in(px_in, (size_t)n * 2 * sizeof(float)), (size_t)n * 2 * sizeof(float), cudaMemcpyHostToDevice, s));
    if (initial) DSDTM_CUDA(c, cudaMemcpyAsync(c->lift_initial_d, st.in(initial, (size_t)n), (size_t)n, cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_INGEST);
    DSDTM_CUDA(c, launch_keyframe_lift(c, depth_slot, pose_c2w, dist, depth_slot >= 0 ? depth_scale : 1.0f, initial != nullptr, n, s));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(out, (size_t)n * sizeof(dsdtm_lifted)), c->lift_out_d, (size_t)n * sizeof(dsdtm_lifted), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    st.finish();
    return 0;
}

// Device-resident map table + Tracking::GetCloseKeyFrames / UpdateLocalMap ranking (ref: src/Tracking.cpp:261-277,315-345)
int dsdtm_map_table_upload(dsdtm_ctx* c, int first_kf, int n_kfs, const dsdtm_map_kf* kfs, int first_point, int n_points, const double* points_w)
{
    if (!c) return DSDTM_E_ARG;
    if (first_kf < 0 || n_kfs < 0 || first_point < 0 || n_points < 0) return fail(c, DSDTM_E_ARG, "negative range");
    if ((n_kfs && !kfs) || (n_points && !points_w)) return fail(c, DSDTM_E_ARG, "null pointer");
    if ((size_t)first_kf > c->mt_kfs_n || (size_t)first_point > c->mt_pts_n) return fail(c, DSDTM_E_ARG, "range starts past the end of the table (rows are appended or rewritten, never skipped)");
    const size_t end_kf = (size_t)first_kf + n_kfs, end_pt = (size_t)first_point + n_points;
    const size_t pts_after = std::max(c->mt_pts_n, end_pt);
    for (int k = 0; k < n_kfs; ++k)
        if (kfs[k].pt_begin < 0 || kfs[k].pt_count < 0 || (size_t)kfs[k].pt_begin + kfs[k].pt_count > pts_after)
            return fail(c, DSDTM_E_ARG, "key-frame row points outside the point array");
    if (grow_keep(c, &c->mt_kfs_d, &c->mt_kfs_cap, end_kf, c->mt_kfs_n) || grow_keep(c, &c->mt_pts_d, &c->mt_pts_cap, 3 * end_pt, 3 * c->mt_pts_n))
        return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    Stager st(c, (size_t)n_kfs * sizeof(dsdtm_map_kf) + 3 * (size_t)n_points * sizeof(double));
    if (n_kfs) DSDTM_CUDA(c, cudaMemcpyAsync(c->mt_kfs_d + first_kf, st.in(kfs, (size_t)n_kfs * sizeof(dsdtm_map_kf)), (size_t)n_kfs * sizeof(dsdtm_map_kf), cudaMemcpyHostToDevice, s));
    if (n_points) DSDTM_CUDA(c, cudaMemcpyAsync(c->mt_pts_d + 3 * (size_t)first_point, st.in(points_w, 3 * (size_t)n_points * sizeof(double)), 3 * (size_t)n_points * sizeof(double), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));     // the caller's buffers may go away
    c->mt_kfs_n = std::max(c->mt_kfs_n, end_kf);
    c->mt_pts_n = pts_after;
    return 0;
}

int dsdtm_close_keyframes(dsdtm_ctx* c, const double pose_cur_c2w[7], int n_kfs, int max_local, uint8_t* visible, double* dist,
                          int32_t* local, int32_t* n_local)
{
    if (!c || !pose_cur_c2w || !n_local || n_kfs < 0 || max_local < 0 || (max_local && !local)) return DSDTM_E_ARG;
    if ((size_t)n_kfs > c->mt_kfs_n) return fail(c, DSDTM_E_ARG, "n_kfs exceeds the uploaded map table");
    *n_local = 0;
    if (n_kfs == 0) return 0;
    if (grow(c, &c->mt_vis_d, &c->mt_vis_cap, (size_t)n_kfs) || grow(c, &c->mt_dist_d, &c->mt_dist_cap, (size_t)n_kfs)) return DSDTM_E_NOMEM;
    if (ensure_pinned(c, (size_t)n_kfs * (sizeof(double) + 1) + 16)) return DSDTM_E_NOMEM;
    double* dist_h = reinterpret_cast<double*>(c->pinned);
    uint8_t* vis_h = c->pinned + (size_t)n_kfs * sizeof(double);
    cudaStream_t s = c->stream;
    stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
    DSDTM_CUDA(c, launch_close_keyframes(c, pose_cur_c2w, n_kfs, s));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(dist_h, c->mt_dist_d, (size_t)n_kfs * sizeof(double), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(vis_h, c->mt_vis_d, (size_t)n_kfs, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    if (visible) std::memcpy(visible, vis_h, (size_t)n_kfs);
    if (dist) std::memcpy(dist, dist_h, (size_t)n_kfs * sizeof(double));
    // UpdateLocalMap's ranking (ref: src/Tracking.cpp:266-277): stable sort of the close key frames by distance, first max_local
    std::vector<int32_t> order;
    for (int k = 0; k < n_kfs; ++k) if (vis_h[k]) order.push_back(k);
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return dist_h[a] < dist_h[b]; });
    const int n = std::min<int>((int)order.size(), max_local);
    for (int i = 0; i < n; ++i) local[i] = order[i];
    *n_local = n;
    return 0;
}

// ------------------------------------------------------------------------------------------------ device-resident map store
int dsdtm_store_clear(dsdtm_ctx* c)
{
    if (!c) return DSDTM_E_ARG;
    c->st_kfs_n = c->st_feats_n = c->st_pts_n = 0;
    c->st_max_feats = 0;
    c->st_kf_nfeat.clear();
    c->st_kf_slot.clear();
    c->batch.commit_flags = 0; c->batch.advance_flags = 0;                   // the step's matches name rows that are gone
    drop_store_graphs(c);
    return 0;
}

int dsdtm_store_set_points(dsdtm_ctx* c, int first, int n, const double* point_w, const int32_t* bad)
{
    if (!c) return DSDTM_E_ARG;
    if (first < 0 || n < 0 || (n && !point_w)) return fail(c, DSDTM_E_ARG, "dsdtm_store_set_points: bad range / null positions");
    if ((size_t)first > c->st_pts_n) return fail(c, DSDTM_E_ARG, "dsdtm_store_set_points: range starts past the end (points are appended or rewritten)");
    if (n == 0) return 0;
    drop_store_graphs(c);
    const size_t end = (size_t)first + n, old_n = c->st_pts_n;
    const size_t old_claim_cap = c->st_claim_cap;
    if (grow_keep(c, &c->st_pts_d, &c->st_pts_cap, end, old_n) || grow_keep(c, &c->st_claim_d, &c->st_claim_cap, end, old_n) ||
        grow_keep(c, &c->st_found_d, &c->st_found_cap, end, old_n)) return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    if (c->st_claim_cap != old_claim_cap)     // fresh part of the claim array: "never claimed"
        DSDTM_CUDA(c, cudaMemsetAsync(c->st_claim_d + old_n, 0xFF, (c->st_claim_cap - old_n) * sizeof(unsigned long long), s));
    std::vector<dsdtm_store_point> rows((size_t)n);
    std::vector<int32_t> last((size_t)n, -1);
    const size_t n_old = end > old_n ? (old_n > (size_t)first ? old_n - first : 0) : (size_t)n;   // rows that already exist keep their chains
    if (n_old) {
        std::vector<dsdtm_store_point> cur(n_old);
        DSDTM_CUDA(c, cudaMemcpyAsync(cur.data(), c->st_pts_d + first, n_old * sizeof(dsdtm_store_point), cudaMemcpyDeviceToHost, s));
        DSDTM_CUDA(c, cudaStreamSynchronize(s));
        for (size_t i = 0; i < n_old; ++i) last[i] = cur[i].last_obs;
    }
    for (int i = 0; i < n; ++i) {
        for (int k = 0; k < 3; ++k) rows[(size_t)i].point_w[k] = point_w[3 * (size_t)i + k];
        rows[(size_t)i].bad = bad ? bad[i] : 0;
        rows[(size_t)i].last_obs = last[(size_t)i];
    }
    DSDTM_CUDA(c, cudaMemcpyAsync(c->st_pts_d + first, rows.data(), (size_t)n * sizeof(dsdtm_store_point), cudaMemcpyHostToDevice, s));
    const std::vector<int32_t> ones(end > old_n ? end - old_n : 0, 1);                            // MapPoint::mnFound starts at 1
    if (!ones.empty()) DSDTM_CUDA(c, cudaMemcpyAsync(c->st_found_d + old_n, ones.data(), ones.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    c->st_pts_n = std::max(old_n, end);
    return 0;
}

namespace {
__global__ void store_update_points_kernel(dsdtm_store_point* pts, const int32_t* ids, int n, const double* pw, const int32_t* bad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    dsdtm_store_point& p = pts[ids[i]];
    if (pw) { p.point_w[0] = pw[3 * i]; p.point_w[1] = pw[3 * i + 1]; p.point_w[2] = pw[3 * i + 2]; }
    if (bad) p.bad = bad[i];
}
}  // namespace

int dsdtm_store_update_points(dsdtm_ctx* c, const int32_t* ids, int n, const double* point_w, const int32_t* bad)
{
    if (!c) return DSDTM_E_ARG;
    if (n < 0 || (n && !ids)) return fail(c, DSDTM_E_ARG, "dsdtm_store_update_points: null ids");
    if (n == 0 || (!point_w && !bad)) return 0;
    for (int i = 0; i < n; ++i) if (ids[i] < 0 || (size_t)ids[i] >= c->st_pts_n) return fail(c, DSDTM_E_ARG, "dsdtm_store_update_points: id outside the point table");
    drop_store_graphs(c);
    const int chunk = 16384;                                     // 16384 x 32 B + padding fits the 1 MB staging mirror
    cudaStream_t s = c->stream;
    for (int i0 = 0; i0 < n; i0 += chunk) {
        const int m = std::min(chunk, n - i0);
        size_t off = 0;
        auto up = [&](const void* src, size_t nb) -> void* {
            std::memcpy(c->stage_pin + off, src, nb);
            void* dst = c->stage_dev + off;
            cudaMemcpyAsync(dst, c->stage_pin + off, nb, cudaMemcpyHostToDevice, s);
            off += (nb + 15) & ~(size_t)15;
            return dst;
        };
        const double* pw_d = point_w ? static_cast<const double*>(up(point_w + 3 * (size_t)i0, (size_t)m * 3 * sizeof(double))) : nullptr;
        const int32_t* ids_d = static_cast<const int32_t*>(up(ids + i0, (size_t)m * sizeof(int32_t)));
        const int32_t* bad_d = bad ? static_cast<const int32_t*>(up(bad + i0, (size_t)m * sizeof(int32_t))) : nullptr;
        store_update_points_kernel<<<(m + 127) / 128, 128, 0, s>>>(c->st_pts_d, ids_d, m, pw_d, bad_d);
        c->launches++;
        DSDTM_CUDA(c, cudaGetLastError());
        DSDTM_CUDA(c, cudaStreamSynchronize(s));                 // the staging arena is reused by the next chunk / call
    }
    return 0;
}

int dsdtm_store_append_keyframe(dsdtm_ctx* c, const dsdtm_store_kf* kf, const dsdtm_store_feat* feats, int n_feats, int32_t* row)
{
    if (!c || !kf) return DSDTM_E_ARG;
    if (n_feats < 0 || (n_feats && !feats) || n_feats > 65535) return fail(c, DSDTM_E_ARG, "dsdtm_store_append_keyframe: bad feature count");
    if (check_slot(c, kf->slot)) return DSDTM_E_ARG;
    for (int j = 0; j < n_feats; ++j)
        if (feats[j].mp >= (int)c->st_pts_n || feats[j].level < 0 || feats[j].level >= c->geo.levels)
            return fail(c, DSDTM_E_ARG, "dsdtm_store_append_keyframe: feature names a map point outside the point table (append the points first) or a bad level");
    drop_store_graphs(c);
    const size_t r = c->st_kfs_n, f0 = c->st_feats_n;
    if (grow_keep(c, &c->st_kfs_d, &c->st_kfs_cap, r + 1, r) || grow_keep(c, &c->st_feats_d, &c->st_feats_cap, f0 + n_feats, f0)) return DSDTM_E_NOMEM;
    if (grow(c, &c->st_vis_d, &c->st_vis_cap, r + 1) || grow(c, &c->st_dist_d, &c->st_dist_cap, r + 1)) return DSDTM_E_NOMEM;
    if (!c->st_sel_d && dalloc(c, &c->st_sel_d, 32)) return DSDTM_E_NOMEM;
    dsdtm_store_kf k = *kf;
    k.feat_begin = (int32_t)f0; k.feat_count = n_feats;
    std::vector<dsdtm_store_feat> fs(feats, feats + n_feats);
    for (auto& f : fs) { f.is_obs = (f.mp >= 0 && f.is_obs) ? (int32_t)r + 1 : 0; f.next_obs = -1; }   // the observing key frame's row + 1
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->st_kfs_d + r, &k, sizeof k, cudaMemcpyHostToDevice, s));
    if (n_feats) DSDTM_CUDA(c, cudaMemcpyAsync(c->st_feats_d + f0, fs.data(), (size_t)n_feats * sizeof(dsdtm_store_feat), cudaMemcpyHostToDevice, s));
    c->st_kfs_n = r + 1; c->st_feats_n = f0 + n_feats;
    c->st_max_feats = std::max(c->st_max_feats, n_feats);
    c->st_kf_nfeat.push_back(n_feats);
    c->st_kf_slot.push_back(kf->slot);
    DSDTM_CUDA(c, launch_store_link(c, (int)f0, n_feats, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    if (row) *row = (int32_t)r;
    return 0;
}

int dsdtm_store_set_keyframe(dsdtm_ctx* c, int row, int slot, const double pose_c2w[7], const double center[3])
{
    if (!c || !pose_c2w || !center) return DSDTM_E_ARG;
    if (row < 0 || (size_t)row >= c->st_kfs_n) return fail(c, DSDTM_E_ARG, "dsdtm_store_set_keyframe: row outside the table");
    if (check_slot(c, slot)) return DSDTM_E_ARG;
    drop_store_graphs(c);
    cudaStream_t s = c->stream;
    dsdtm_store_kf k;
    DSDTM_CUDA(c, cudaMemcpyAsync(&k, c->st_kfs_d + row, sizeof k, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    k.slot = slot;
    for (int i = 0; i < 7; ++i) k.pose_c2w[i] = pose_c2w[i];
    for (int i = 0; i < 3; ++i) k.center[i] = center[i];
    DSDTM_CUDA(c, cudaMemcpyAsync(c->st_kfs_d + row, &k, sizeof k, cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    c->st_kf_slot[(size_t)row] = slot;
    return 0;
}

namespace {
__global__ void store_set_found_kernel(int* found, const int32_t* ids, int n, const int32_t* v)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) found[ids[i]] = v[i];
}
}  // namespace

int dsdtm_store_set_found(dsdtm_ctx* c, const int32_t* ids, int n, const int32_t* found)
{
    if (!c) return DSDTM_E_ARG;
    if (n < 0 || (n && (!ids || !found))) return fail(c, DSDTM_E_ARG, "dsdtm_store_set_found: null ids / counts");
    if (n == 0) return 0;
    for (int i = 0; i < n; ++i) if (ids[i] < 0 || (size_t)ids[i] >= c->st_pts_n) return fail(c, DSDTM_E_ARG, "dsdtm_store_set_found: id outside the point table");
    drop_store_graphs(c);
    const int chunk = 65536;                                     // 2 x 256 KB fits the 1 MB staging mirror
    cudaStream_t s = c->stream;
    for (int i0 = 0; i0 < n; i0 += chunk) {
        const int m = std::min(chunk, n - i0);
        const size_t nb = (size_t)m * sizeof(int32_t);
        std::memcpy(c->stage_pin, ids + i0, nb);
        std::memcpy(c->stage_pin + nb, found + i0, nb);
        DSDTM_CUDA(c, cudaMemcpyAsync(c->stage_dev, c->stage_pin, 2 * nb, cudaMemcpyHostToDevice, s));
        const int32_t* ids_d = reinterpret_cast<const int32_t*>(c->stage_dev);
        store_set_found_kernel<<<(m + 127) / 128, 128, 0, s>>>(c->st_found_d, ids_d, m, ids_d + m);
        c->launches++;
        DSDTM_CUDA(c, cudaGetLastError());
        DSDTM_CUDA(c, cudaStreamSynchronize(s));                 // the staging arena is reused by the next chunk / call
    }
    return 0;
}

int dsdtm_store_size(const dsdtm_ctx* c, int32_t* n_kfs, int32_t* n_feats, int32_t* n_points)
{
    if (!c) return DSDTM_E_ARG;
    if (n_kfs) *n_kfs = (int32_t)c->st_kfs_n;
    if (n_feats) *n_feats = (int32_t)c->st_feats_n;
    if (n_points) *n_points = (int32_t)c->st_pts_n;
    return 0;
}

int dsdtm_store_fetch(dsdtm_ctx* c, int kf_first, int n_kfs, dsdtm_store_kf* kfs, int feat_first, int n_feats, dsdtm_store_feat* feats,
                      int point_first, int n_points, dsdtm_store_point* points, int32_t* found)
{
    if (!c) return DSDTM_E_ARG;
    auto bad_range = [](int first, int n, size_t size) { return first < 0 || n < 0 || (size_t)first + (size_t)n > size; };
    if (bad_range(kf_first, n_kfs, c->st_kfs_n) || bad_range(feat_first, n_feats, c->st_feats_n) || bad_range(point_first, n_points, c->st_pts_n))
        return fail(c, DSDTM_E_ARG, "dsdtm_store_fetch: range outside the store");
    cudaStream_t s = c->stream;
    if (kfs && n_kfs) DSDTM_CUDA(c, cudaMemcpyAsync(kfs, c->st_kfs_d + kf_first, (size_t)n_kfs * sizeof(dsdtm_store_kf), cudaMemcpyDeviceToHost, s));
    if (feats && n_feats) DSDTM_CUDA(c, cudaMemcpyAsync(feats, c->st_feats_d + feat_first, (size_t)n_feats * sizeof(dsdtm_store_feat), cudaMemcpyDeviceToHost, s));
    if (points && n_points) DSDTM_CUDA(c, cudaMemcpyAsync(points, c->st_pts_d + point_first, (size_t)n_points * sizeof(dsdtm_store_point), cudaMemcpyDeviceToHost, s));
    if (found && n_points) DSDTM_CUDA(c, cudaMemcpyAsync(found, c->st_found_d + point_first, (size_t)n_points * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

int dsdtm_store_track(dsdtm_ctx* c, int cur_slot, const double pose_cur_c2w[7], const double cur_center[3], int max_local,
                      int max_search_level, int align_iters, int32_t* local_rows, int32_t* n_local, dsdtm_store_cand* out, int cap,
                      int32_t* n_out)
{
    if (!c || !pose_cur_c2w || !cur_center || !local_rows || !n_local || !n_out || (cap && !out)) return DSDTM_E_ARG;
    if (check_slot(c, cur_slot)) return DSDTM_E_ARG;
    if (max_local < 1 || max_local > 16) return fail(c, DSDTM_E_ARG, "dsdtm_store_track: max_local must be 1..16");
    if (max_search_level < 0 || max_search_level >= c->geo.levels || align_iters < 0) return fail(c, DSDTM_E_ARG, "dsdtm_store_track: bad max_search_level / align_iters");
    const size_t room = (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1);
    if (cap < 0 || (size_t)cap > room) return fail(c, DSDTM_E_ARG, "dsdtm_store_track: cap exceeds max_batch * max_patches");
    *n_local = 0; *n_out = 0;
    if (c->st_kfs_n == 0 || cap == 0) return 0;
    if (grow(c, &c->st_out_d, &c->st_out_cap, (size_t)cap)) return DSDTM_E_NOMEM;
    const size_t out_bytes = (size_t)cap * sizeof(dsdtm_store_cand);
    if (ensure_pinned(c, out_bytes + 32 * sizeof(int))) return DSDTM_E_NOMEM;
    int* sel_h = reinterpret_cast<int*>(c->pinned);
    dsdtm_store_cand* out_h = reinterpret_cast<dsdtm_store_cand*>(c->pinned + 32 * sizeof(int));
    cudaStream_t s = c->stream;
    ++c->st_epoch;
    StoreTrackArgs a;
    a.cur_slot = cur_slot; a.n_kfs = (int)c->st_kfs_n; a.max_local = max_local; a.cap = cap;
    for (int k = 0; k < 7; ++k) a.pose_cur[k] = pose_cur_c2w[k];
    for (int k = 0; k < 3; ++k) a.cur_center[k] = cur_center[k];
    a.max_search_level = max_search_level;
    stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
    DSDTM_CUDA(c, launch_store_track(c, a, s));
    stage_end(c, 2);
    // the record count is only known on the device: warp / Align2D take it from there and skip what lies beyond
    stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
    DSDTM_CUDA(c, launch_warp_affine(c, cap, c->patches_d, s, 0, store_count_dev(c)));
    stage_end(c, 1);
    stage_begin(c, DSDTM_STAGE_ALIGN2D);
    DSDTM_CUDA(c, launch_align2d(c, cap, align_iters, s, 0, store_count_dev(c), c->st_out_d));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(sel_h, c->st_sel_d, 18 * sizeof(int), cudaMemcpyDeviceToHost, s));
    // typical frames have ~1 k candidates: the first copy takes that many, a second one follows only for a fuller frame
    const int first = std::min(cap, 1280);
    DSDTM_CUDA(c, cudaMemcpyAsync(out_h, c->st_out_d, (size_t)first * sizeof(dsdtm_store_cand), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    const int n = sel_h[17], got = std::min(n, cap);
    if (got > first) {
        DSDTM_CUDA(c, cudaMemcpyAsync(out_h + first, c->st_out_d + first, (size_t)(got - first) * sizeof(dsdtm_store_cand), cudaMemcpyDeviceToHost, s));
        DSDTM_CUDA(c, cudaStreamSynchronize(s));
    }
    *n_local = sel_h[0];
    for (int i = 0; i < sel_h[0]; ++i) local_rows[i] = sel_h[1 + i];
    std::memcpy(out, out_h, (size_t)got * sizeof(dsdtm_store_cand));
    *n_out = n;
    if (n > cap) return fail(c, DSDTM_E_ARG, "dsdtm_store_track: more candidates than cap (records truncated)");
    return 0;
}

// Sprase_ImgAlign::Run and Tracking::UpdateLocalMap (+ the arithmetic of SearchLocalPoints) as ONE submission: the pose found by the
// sparse alignment is composed with the reference pose on the device and handed to the map-store kernels through device memory,
// so the frame costs one synchronisation instead of two (ref: src/Tracking.cpp:199-224,257-313).
int dsdtm_track_frame_store(dsdtm_ctx* c, const dsdtm_track_store_in* in, dsdtm_track_out* out, int32_t* local_rows, int32_t* n_local,
                            dsdtm_store_cand* cands, int cap, int32_t* n_out)
{
    if (!c || !in || !out || !in->feats || !local_rows || !n_local || !n_out || (cap && !cands)) return DSDTM_E_ARG;
    const int nf = in->n_feats;
    if (nf < 1 || nf > c->prm.max_feats) return fail(c, DSDTM_E_ARG, "n_feats out of range (max_feats)");
    if (check_pairs(c, 1, &in->ref_slot, &in->cur_slot, nf, &nf, in->max_level, in->min_level, in->max_iters)) return DSDTM_E_ARG;
    if (in->max_local < 1 || in->max_local > 16) return fail(c, DSDTM_E_ARG, "max_local must be 1..16");
    if (in->max_search_level < 0 || in->max_search_level >= c->geo.levels || in->align_iters < 0) return fail(c, DSDTM_E_ARG, "bad max_search_level / align_iters");
    const size_t room = (size_t)c->prm.max_batch * std::max(c->prm.max_patches, 1);
    if (cap < 0 || (size_t)cap > room) return fail(c, DSDTM_E_ARG, "cap exceeds max_batch * max_patches");
    *n_local = 0; *n_out = 0;
    const bool with_map = c->st_kfs_n > 0 && cap > 0;
    if (with_map && grow(c, &c->st_out_d, &c->st_out_cap, (size_t)cap)) return DSDTM_E_NOMEM;
    if (ensure_pinned(c, (size_t)std::max(cap, 1) * sizeof(dsdtm_store_cand) + 32 * sizeof(int))) return DSDTM_E_NOMEM;
    Arena ar(c, 3 * sizeof(int) + 10 * sizeof(double) + (size_t)nf * sizeof(dsdtm_ref_feat), (7 + 10) * sizeof(double) + 2 * sizeof(int), 6, 4);
    if (!ar.active) return fail(c, DSDTM_E_ARG, "dsdtm_track_frame_store: inputs exceed the 1 MB staging arena");
    c->batch.staged = false;
    cudaStream_t s = c->stream;
    PtrSwap<int> p0(c->ref_slots_d, ar.in(&in->ref_slot, 1)), p1(c->cur_slots_d, ar.in(&in->cur_slot, 1)), p2(c->n_feats_d, ar.in(&nf, 1));
    PtrSwap<double> p3(c->centers_d, ar.in(in->ref_center, 3)), p4(c->poses_in_d, ar.in(in->pose_c2r_in, 7));
    PtrSwap<dsdtm_ref_feat> p5(c->feats_d, ar.in(in->feats, (size_t)nf));
    double* pose_c2r_d = ar.out(out->pose_c2r, 7);
    double* pose10_d = ar.out((double*)nullptr, 10);
    PtrSwap<double> q0(c->poses_out_d, pose_c2r_d);
    PtrSwap<int> q1(c->n_tracked_d, ar.out(&out->n_tracked, 1)), q2(c->n_log_d, ar.out((int*)nullptr, 1));
    DSDTM_CUDA(c, ar.upload(s));
    stage_begin(c, DSDTM_STAGE_SPARSE_ALIGN);
    DSDTM_CUDA(c, launch_sparse_align(c, 1, nf, in->max_level, in->min_level, in->max_iters, false, s));
    stage_end(c, 1);
    int* sel_h = reinterpret_cast<int*>(c->pinned);
    dsdtm_store_cand* out_h = reinterpret_cast<dsdtm_store_cand*>(c->pinned + 32 * sizeof(int));
    const int first = std::min(cap, 1280);
    if (!with_map) {
        stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
        DSDTM_CUDA(c, launch_compose_pose(c, pose_c2r_d, in->pose_ref_c2w, pose10_d, s));
        stage_end(c, 1);
    } else {
        ++c->st_epoch;
        StoreTrackArgs a;
        a.cur_slot = in->cur_slot; a.n_kfs = (int)c->st_kfs_n; a.max_local = in->max_local; a.cap = cap;
        for (int k = 0; k < 7; ++k) a.pose_cur[k] = 0.0;
        for (int k = 0; k < 3; ++k) a.cur_center[k] = 0.0;
        a.t_c2r_dev = pose_c2r_d; a.pose10_out = pose10_d;
        for (int k = 0; k < 7; ++k) a.pose_ref[k] = in->pose_ref_c2w[k];
        a.max_search_level = in->max_search_level;
        stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
        DSDTM_CUDA(c, launch_store_track(c, a, s));
        stage_end(c, 2);
        stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
        DSDTM_CUDA(c, launch_warp_affine(c, cap, c->patches_d, s, 0, store_count_dev(c)));
        stage_end(c, 1);
        stage_begin(c, DSDTM_STAGE_ALIGN2D);
        DSDTM_CUDA(c, launch_align2d(c, cap, in->align_iters, s, 0, store_count_dev(c), c->st_out_d));
        stage_end(c, 1);
        DSDTM_CUDA(c, cudaMemcpyAsync(sel_h, c->st_sel_d, 18 * sizeof(int), cudaMemcpyDeviceToHost, s));
        DSDTM_CUDA(c, cudaMemcpyAsync(out_h, c->st_out_d, (size_t)first * sizeof(dsdtm_store_cand), cudaMemcpyDeviceToHost, s));
    }
    DSDTM_CUDA(c, ar.download(s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    ar.finish();
    const double* p10 = ar.host_view(pose10_d);
    for (int k = 0; k < 7; ++k) out->pose_cur_c2w[k] = p10[k];
    for (int k = 0; k < 3; ++k) out->cur_center[k] = p10[7 + k];
    out->reserved = 0;
    if (with_map) {
        const int n = sel_h[17], got = std::min(n, cap);
        if (got > first) {
            DSDTM_CUDA(c, cudaMemcpyAsync(out_h + first, c->st_out_d + first, (size_t)(got - first) * sizeof(dsdtm_store_cand), cudaMemcpyDeviceToHost, s));
            DSDTM_CUDA(c, cudaStreamSynchronize(s));
        }
        *n_local = sel_h[0];
        for (int i = 0; i < sel_h[0]; ++i) local_rows[i] = sel_h[1 + i];
        std::memcpy(cands, out_h, (size_t)got * sizeof(dsdtm_store_cand));
        *n_out = n;
        if (n > cap) return fail(c, DSDTM_E_ARG, "dsdtm_track_frame_store: more candidates than cap (records truncated)");
    }
    return 0;
}

// Optimizer::PoseOptimization (ref: src/Optimizer.cpp:20-101) for n_frames independent frames: one copy in per array, one launch,
// one copy out per requested array, one synchronisation.
int dsdtm_pose_optimize_batch(dsdtm_ctx* c, int n_frames, const dsdtm_ba_obs* obs, int obs_stride, const int* n_obs,
                              const double* poses_in, int max_iters, double* poses_out, double* res_norm, dsdtm_ba_summary* summaries)
{
    if (!c) return DSDTM_E_ARG;
    if (n_frames < 0 || obs_stride < 0 || max_iters < 0) return fail(c, DSDTM_E_ARG, "negative count");
    if (n_frames == 0) return 0;
    if (!n_obs || !poses_in || !poses_out) return fail(c, DSDTM_E_ARG, "null pointer");
    int max_obs = 0;
    for (int i = 0; i < n_frames; ++i) {
        if (n_obs[i] < 0 || n_obs[i] > obs_stride) return fail(c, DSDTM_E_ARG, "n_obs outside [0, obs_stride]");
        max_obs = std::max(max_obs, n_obs[i]);
    }
    if (max_obs > DSDTM_BA_MAX_OBS) return fail(c, DSDTM_E_ARG, "more than DSDTM_BA_MAX_OBS observations in a frame");
    if (max_obs > 0 && !obs) return fail(c, DSDTM_E_ARG, "null pointer");
    for (int i = 0; i < n_frames; ++i)
        for (int k = 0; k < n_obs[i]; ++k) {
            const int L = obs[(size_t)i * obs_stride + k].level;
            if (L < 0 || L > 30) return fail(c, DSDTM_E_ARG, "observation level outside [0, 30]");
        }
    const size_t n_rec = (size_t)n_frames * obs_stride;
    {
        // small calls (one frame, a few frames): everything in ONE copy each way through the pinned arena and its device mirror
        const size_t nf = (size_t)n_frames;
        Arena ar(c, n_rec * sizeof(dsdtm_ba_obs) + nf * (sizeof(int) + 7 * sizeof(double)),
                 nf * (7 * sizeof(double) + sizeof(dsdtm_ba_summary)) + (res_norm ? n_rec * sizeof(double) : 0), 3, 3);
        if (ar.active) {
            cudaStream_t s = c->stream;
            dsdtm_ba_obs* dummy_obs = nullptr;
            PtrSwap<dsdtm_ba_obs> p0(c->po_obs_d, n_rec ? ar.in(obs, n_rec) : dummy_obs);
            PtrSwap<int> p1(c->po_nobs_d, ar.in(n_obs, nf));
            PtrSwap<double> p2(c->po_pose_in_d, ar.in(poses_in, 7 * nf)), q0(c->po_pose_out_d, ar.out(poses_out, 7 * nf));
            PtrSwap<dsdtm_ba_summary> q1(c->po_sum_d, ar.out(summaries, nf));
            PtrSwap<double> q2(c->po_res_d, (res_norm && n_rec) ? ar.out(res_norm, n_rec) : c->po_res_d);
            DSDTM_CUDA(c, ar.upload(s));
            stage_begin(c, DSDTM_STAGE_POSE_OPT);
            DSDTM_CUDA(c, launch_pose_opt(c, n_frames, obs_stride, max_obs, max_iters, res_norm != nullptr && n_rec, summaries != nullptr, s));
            stage_end(c, 1);
            DSDTM_CUDA(c, ar.download(s));
            DSDTM_CUDA(c, cudaStreamSynchronize(s));
            ar.finish();
            return 0;
        }
    }
    if (grow(c, &c->po_obs_d, &c->po_obs_cap, n_rec) || grow(c, &c->po_nobs_d, &c->po_nobs_cap, (size_t)n_frames) ||
        grow(c, &c->po_pose_in_d, &c->po_pose_in_cap, 7 * (size_t)n_frames) || grow(c, &c->po_pose_out_d, &c->po_pose_out_cap, 7 * (size_t)n_frames) ||
        grow(c, &c->po_sum_d, &c->po_sum_cap, (size_t)n_frames) || (res_norm && grow(c, &c->po_res_d, &c->po_res_cap, n_rec)))
        return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    Stager st(c, n_rec * (sizeof(dsdtm_ba_obs) + (res_norm ? sizeof(double) : 0)) + (size_t)n_frames * (sizeof(int) + 14 * sizeof(double) + sizeof(dsdtm_ba_summary)));
    if (n_rec) DSDTM_CUDA(c, cudaMemcpyAsync(c->po_obs_d, st.in(obs, n_rec * sizeof(dsdtm_ba_obs)), n_rec * sizeof(dsdtm_ba_obs), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->po_nobs_d, st.in(n_obs, (size_t)n_frames * sizeof(int)), (size_t)n_frames * sizeof(int), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->po_pose_in_d, st.in(poses_in, 7 * (size_t)n_frames * sizeof(double)), 7 * (size_t)n_frames * sizeof(double), cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_POSE_OPT);
    DSDTM_CUDA(c, launch_pose_opt(c, n_frames, obs_stride, max_obs, max_iters, res_norm != nullptr, summaries != nullptr, s));
    stage_end(c, 1);
    DSDTM_CUDA(c, cudaMemcpyAsync(st.out(poses_out, 7 * (size_t)n_frames * sizeof(double)), c->po_pose_out_d, 7 * (size_t)n_frames * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (res_norm && n_rec) DSDTM_CUDA(c, cudaMemcpyAsync(st.out(res_norm, n_rec * sizeof(double)), c->po_res_d, n_rec * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (summaries) DSDTM_CUDA(c, cudaMemcpyAsync(st.out(summaries, (size_t)n_frames * sizeof(dsdtm_ba_summary)), c->po_sum_d, (size_t)n_frames * sizeof(dsdtm_ba_summary), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    st.finish();
    return 0;
}

int dsdtm_pose_optimize(dsdtm_ctx* c, const dsdtm_ba_obs* obs, int n_obs, const double pose_in[7], int max_iters, double pose_out[7],
                        double* res_norm, dsdtm_ba_summary* summary)
{
    return dsdtm_pose_optimize_batch(c, 1, obs, n_obs, &n_obs, pose_in, max_iters, pose_out, res_norm, summary);
}

int dsdtm_frames_upload_clahe_pyramid(dsdtm_ctx* c, int first_slot, int n, const uint8_t* imgs, double clip_limit, int tiles_x, int tiles_y,
                                      uint8_t* level0_out)
{
    if (!c || !imgs || n < 0) return DSDTM_E_ARG;
    if (n == 0) return 0;
    if (check_slot(c, first_slot, n) || check_grid_frames(c, n)) return DSDTM_E_ARG;
    const LevelGeom& g = c->geo;
    const int w = g.w[0], h = g.h[0];
    if (tiles_x < 1 || tiles_y < 1 || tiles_x > clahe_max_tiles_x() || w % tiles_x || h % tiles_y)
        return fail(c, DSDTM_E_ARG, "CLAHE: the image size must be divisible by the tile grid, tiles_x <= 16");
    if (h / tiles_y < clahe_rows_per_cta()) return fail(c, DSDTM_E_ARG, "CLAHE: tile height must be >= 8");
    const size_t px = (size_t)w * h, lut = (size_t)tiles_x * tiles_y * 256;
    if (grow(c, &c->clahe_src_d, &c->clahe_cap, px * n) || grow(c, &c->clahe_lut_d, &c->clahe_lut_cap, lut * n)) return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->clahe_src_d, imgs, px * n, cudaMemcpyHostToDevice, s));
    stage_begin(c, DSDTM_STAGE_INGEST);
    DSDTM_CUDA(c, launch_clahe(c, first_slot, n, clip_limit, tiles_x, tiles_y, s));
    stage_end(c, 2);
    stage_begin(c, DSDTM_STAGE_PYRAMID);
    DSDTM_CUDA(c, launch_pyramid(c, first_slot, n, s));
    stage_end(c, pyramid_launches(c));
    if (level0_out)
        DSDTM_CUDA(c, cudaMemcpy2DAsync(level0_out, px, c->frames_d + (size_t)first_slot * g.frame_stride + g.off[0], g.frame_stride, px, n,
                                        cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

// ------------------------------------------------------------------------------------------------ batched front end
static int stage_patches(dsdtm_ctx* c, int n_pairs, const int* cur_slots, const uint8_t* patches10, const double* patch_px,
                         const int* patch_level, int ppp, cudaStream_t s, int pair0 = 0)
{
    if (ppp <= 0) return 0;
    const size_t n = (size_t)n_pairs * ppp, o = (size_t)pair0 * ppp;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patches_d + o * 100, patches10 + o * 100, n * 100, cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patch_px_in_d + o * 2, patch_px + o * 2, n * 2 * sizeof(double), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->patch_level_d + o, patch_level + o, n * sizeof(int), cudaMemcpyHostToDevice, s));
    return 0;
}

__global__ void fill_patch_slots_kernel(const int* __restrict__ cur_slots, int* __restrict__ patch_slot, int ppp, int n, int o)
{
    const int i = o + blockIdx.x * blockDim.x + threadIdx.x;
    if (i < o + n) patch_slot[i] = cur_slots[i / ppp];
}

int dsdtm_batch_stage(dsdtm_ctx* c, int n_pairs, const int* ref_slots, const int* cur_slots, const dsdtm_ref_feat* feats, int feat_stride,
                      const int* n_feats, const double* ref_centers, const double* poses_in, int max_level, int min_level, int max_iters,
                      const uint8_t* patches10, const double* patch_px, const int* patch_level, int ppp, int align_iters)
{
    if (!c || !ref_slots || !cur_slots || !feats || !n_feats || !ref_centers || !poses_in) return DSDTM_E_ARG;
    if (check_grid_frames(c, n_pairs) || check_pairs(c, n_pairs, ref_slots, cur_slots, feat_stride, n_feats, max_level, min_level, max_iters))
        return DSDTM_E_ARG;
    if (ppp < 0 || ppp > c->prm.max_patches || align_iters < 0) return fail(c, DSDTM_E_ARG, "patches_per_pair > max_patches");
    if (ppp > 0 && (!patches10 || !patch_px || !patch_level)) return fail(c, DSDTM_E_ARG, "null patch arrays");
    cudaStream_t s = c->stream;
    if (stage_pairs(c, n_pairs, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_in, s)) return DSDTM_E_CUDA;
    if (stage_patches(c, n_pairs, cur_slots, patches10, patch_px, patch_level, ppp, s)) return DSDTM_E_CUDA;
    if (ppp > 0) {
        const int n = n_pairs * ppp;
        fill_patch_slots_kernel<<<(n + 255) / 256, 256, 0, s>>>(c->cur_slots_d, c->patch_slot_d, ppp, n, 0);
        DSDTM_CUDA(c, cudaGetLastError());
    }
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    auto& b = c->batch;
    b.staged = true; b.n_pairs = n_pairs; b.feat_stride = feat_stride; b.max_level = max_level; b.min_level = min_level;
    b.max_iters = max_iters; b.patches_per_pair = ppp; b.align_iters = align_iters;
    b.ref_h.assign(ref_slots, ref_slots + n_pairs); b.cur_h.assign(cur_slots, cur_slots + n_pairs);
    b.map_staged = false; b.store_staged = false; b.track_staged = false; b.kf_staged = false; b.commit_flags = 0; b.advance_flags = 0;
    return 0;
}

int dsdtm_batch_stage_map(dsdtm_ctx* c, const double* poses_ref_c2w, int points_per_pair, int max_search_level, int align_iters)
{
    if (!c || !poses_ref_c2w) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_stage_map: call dsdtm_batch_stage first");
    if (points_per_pair < 1 || points_per_pair > c->prm.max_patches || points_per_pair > b.feat_stride)
        return fail(c, DSDTM_E_ARG, "points_per_pair must be 1..min(max_patches, feat_stride)");
    if (max_search_level < 0 || max_search_level >= c->geo.levels || align_iters < 0) return fail(c, DSDTM_E_ARG, "bad max_search_level / align_iters");
    DSDTM_CUDA(c, cudaMemcpyAsync(c->poses_ref_d, poses_ref_c2w, (size_t)b.n_pairs * 7 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    b.map_staged = true; b.map_ppp = points_per_pair; b.max_search_level = max_search_level; b.map_align_iters = align_iters;
    b.store_staged = false; b.track_staged = false; b.kf_staged = false; b.commit_flags = 0; b.advance_flags = 0;
    drop_graphs(c);
    return 0;
}

// prelude CTA of the store-backed chain: the longest range and the table for max_local key frames must fit one CTA's shared memory
static int check_store_batch_smem(dsdtm_ctx* c, int range_len, int max_local, const char* who)
{
    int max_smem = 0;
    DSDTM_CUDA(c, cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
    if (store_batch_smem(c, range_len, max_local) > (size_t)max_smem - 1024) {
        char buf[160];
        snprintf(buf, sizeof buf, "%s: key-frame range and local map beyond one CTA's shared memory", who);
        return fail(c, DSDTM_E_ARG, buf);
    }
    return 0;
}

int dsdtm_batch_stage_store(dsdtm_ctx* c, const double* poses_ref_c2w, const int32_t* kf_range, int max_local, int max_search_level,
                            int align_iters, int cands_per_frame)
{
    if (!c || !poses_ref_c2w) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_stage_store: call dsdtm_batch_stage first");
    if (c->st_kfs_n == 0) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_store: the map store is empty");
    if (max_local < 1 || max_local > 16) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_store: max_local must be 1..16");
    if (cands_per_frame < 1 || cands_per_frame > c->prm.max_patches)
        return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_store: cands_per_frame must be 1..max_patches");
    if (max_search_level < 0 || max_search_level >= c->geo.levels || align_iters < 0)
        return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_store: bad max_search_level / align_iters");
    const int n = b.n_pairs, n_kfs = (int)c->st_kfs_n;
    int range_max = n_kfs, range_end = n_kfs;
    if (kf_range) {
        range_max = 0; range_end = 0;
        for (int i = 0; i < n; ++i) {
            const int k0 = kf_range[2 * i], k1 = kf_range[2 * i + 1];
            if (k0 < 0 || k1 < k0 || k1 > n_kfs) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_store: key-frame range outside the store");
            range_max = std::max(range_max, k1 - k0); range_end = std::max(range_end, k1);
        }
    }
    if (check_store_batch_smem(c, range_max, max_local, "dsdtm_batch_stage_store")) return DSDTM_E_ARG;
    const size_t B = c->prm.max_batch;
    if (!c->sb_rec_d) {
        // once per context at max_batch size: a captured step keeps pointing at these buffers
        if (dalloc(c, &c->sb_rec_d, B * std::max(c->prm.max_patches, 1)) || dalloc(c, &c->sb_ncand_d, B) || dalloc(c, &c->sb_local_d, B * 17) ||
            dalloc(c, &c->sb_pose10_d, B * 10) || dalloc(c, &c->sb_range_d, B))
            return DSDTM_E_NOMEM;
        DSDTM_CUDA(c, store_batch_init(c));
        DSDTM_CUDA(c, track_select_init(c));
    }
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->poses_ref_d, poses_ref_c2w, (size_t)n * 7 * sizeof(double), cudaMemcpyHostToDevice, s));
    if (kf_range) DSDTM_CUDA(c, cudaMemcpyAsync(c->sb_range_d, kf_range, (size_t)n * sizeof(int2), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    b.store_staged = true; b.store_all_rows = kf_range == nullptr; b.store_max_local = max_local; b.store_cpf = cands_per_frame;
    b.store_range_max = range_max; b.store_range_end = range_end;
    b.max_search_level = max_search_level; b.map_align_iters = align_iters;
    b.map_staged = false; b.track_staged = false; b.kf_staged = false; b.commit_flags = 0; b.advance_flags = 0;
    drop_graphs(c);
    return 0;
}

int dsdtm_batch_fetch_store(dsdtm_ctx* c, int32_t* local_rows, int32_t* n_local, dsdtm_store_cand* cands, int32_t* n_cand)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !b.store_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_fetch_store: no staged store batch");
    cudaStream_t s = c->stream;
    const size_t n = (size_t)b.n_pairs, F = (size_t)b.store_cpf;
    std::vector<int32_t> loc(n * 17), nc(n);
    DSDTM_CUDA(c, cudaMemcpyAsync(loc.data(), c->sb_local_d, n * 17 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(nc.data(), c->sb_ncand_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (cands) DSDTM_CUDA(c, cudaMemcpyAsync(cands, c->sb_rec_d, n * F * sizeof(dsdtm_store_cand), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    for (size_t i = 0; i < n; ++i) {
        if (local_rows) for (int r = 0; r < 16; ++r) local_rows[16 * i + r] = loc[17 * i + 1 + r];
        if (n_local) n_local[i] = loc[17 * i];
        // rows past a frame's count hold what earlier replays left there
        const size_t k = std::min((size_t)std::max(nc[i], 0), F);
        if (cands) std::memset(cands + i * F + k, 0, (F - k) * sizeof(dsdtm_store_cand));
    }
    if (n_cand) std::memcpy(n_cand, nc.data(), n * sizeof(int32_t));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->last_run_ms = ms;
    return 0;
}

static int stage_track(dsdtm_ctx* c, const int32_t* found, int max_iters, bool live)
{
    auto& b = c->batch;
    if (live && (!b.staged || !b.store_staged))
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_stage_track_live: call dsdtm_batch_stage_store first");
    if (!b.staged || !(b.map_staged || b.store_staged))
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_stage_track: call dsdtm_batch_stage_map or dsdtm_batch_stage_store first");
    if (max_iters < 0) return fail(c, DSDTM_E_ARG, "negative max_iters");
    if (c->prm.cell_size > track_select_max_radius()) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_track: cell_size above the selection's circle bound");
    if (c->n_cells >= (1 << 22)) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_track: too many grid cells");
    if (b.store_staged && track_select_key_bits(c, b.store_cpf) > 64)
        return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_track: grid cells x cands_per_frame beyond the selection's 64-bit keys");
    if (b.store_staged) {
        int max_smem = 0;
        DSDTM_CUDA(c, cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
        if (track_select_smem(b.store_cpf) > (size_t)max_smem - 1024)
            return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_track: cands_per_frame beyond the selection's shared memory");
    }
    const size_t B = c->prm.max_batch, K = DSDTM_TRACK_MAX_MATCHES;
    if (!c->trk_found_d) {
        // once per context at max_batch size: a captured step keeps pointing at these buffers
        if (dalloc(c, &c->trk_found_d, B * std::max(c->prm.max_patches, 1)) || dalloc(c, &c->trk_match_d, B * K) || dalloc(c, &c->trk_obs_d, B * K) ||
            dalloc(c, &c->trk_nobs_d, B) || dalloc(c, &c->trk_pose_in_d, B * 7) || dalloc(c, &c->trk_pose_out_d, B * 7) ||
            dalloc(c, &c->trk_res_d, B * K) || dalloc(c, &c->trk_sum_d, B))
            return DSDTM_E_NOMEM;
    }
    cudaStream_t s = c->stream;
    // per pair and record, or in store mode per store point row
    const size_t n = b.store_staged ? c->st_pts_n : (size_t)b.n_pairs * b.map_ppp;
    std::vector<int32_t> ones;
    if (!found && !live) { ones.assign(std::max(n, (size_t)1), 1); found = ones.data(); }   // MapPoint::mnFound starts at 1
    if (live) {
        b.store_n_found = 0;                                   // the selection reads the store's own counts (enqueue_track)
    } else if (b.store_staged) {
        if (grow(c, &c->sb_found_d, &c->sb_found_cap, std::max(n, (size_t)1))) return DSDTM_E_NOMEM;
        if (n) DSDTM_CUDA(c, cudaMemcpyAsync(c->sb_found_d, found, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        b.store_n_found = (int)n;
    } else {
        DSDTM_CUDA(c, cudaMemcpyAsync(c->trk_found_d, found, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    }
    // rows past a pair's match count are never written by the step: defined (zero) bytes for the fetch
    DSDTM_CUDA(c, cudaMemsetAsync(c->trk_match_d, 0, B * K * sizeof(dsdtm_match), s));
    DSDTM_CUDA(c, cudaMemsetAsync(c->trk_res_d, 0, B * K * sizeof(double), s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    b.track_staged = true; b.track_iters = max_iters; b.kf_staged = false; b.store_found_live = live; b.commit_flags = 0; b.advance_flags = 0;
    drop_graphs(c);
    return 0;
}

int dsdtm_batch_stage_track(dsdtm_ctx* c, const int32_t* found, int max_iters)
{
    if (!c) return DSDTM_E_ARG;
    return stage_track(c, found, max_iters, false);
}

int dsdtm_batch_stage_track_live(dsdtm_ctx* c, int max_iters)
{
    if (!c) return DSDTM_E_ARG;
    return stage_track(c, nullptr, max_iters, true);
}

int dsdtm_batch_stage_keyframe(dsdtm_ctx* c, const int32_t* depth_slots, const uint8_t* want, float detection_threshold, int min_dist, int max_fts,
                               const float dist[5], float depth_scale)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !(b.map_staged || b.store_staged) || !b.track_staged)
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_stage_keyframe: call dsdtm_batch_stage_track first");
    if (!dist || !(detection_threshold >= 0.f)) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: dist NULL or detection_threshold < 0");
    if (max_fts < 1 || max_fts > DSDTM_MAX_FEATS_LIMIT) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: max_fts must be 1..DSDTM_MAX_FEATS_LIMIT");
    if (min_dist < 0 || min_dist > detect_select_max_radius() || c->prm.cell_size > detect_select_max_radius())
        return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: min_dist / cell_size out of the circle range (0..64)");
    int max_smem = 0;
    DSDTM_CUDA(c, cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
    if (!detect_select_fits(c, (size_t)max_smem))
        return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: frame geometry beyond the selection bitmap (752 x 480 pixels)");
    const int n = b.n_pairs;
    std::vector<int32_t> ds(n, -1);
    std::vector<uint8_t> wt(n, 1);
    bool any_depth = false;
    for (int i = 0; i < n; ++i) {
        if (depth_slots) ds[i] = depth_slots[i];
        if (want) wt[i] = want[i] ? 1 : 0;
        if (ds[i] < -1 || ds[i] >= c->depth_slots) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: depth slot out of range (option depth_slots)");
        if (ds[i] >= 0 && !c->depth_d) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: depth slot given before any depth upload");
        any_depth |= ds[i] >= 0;
    }
    if (any_depth && !(depth_scale > 0.f)) return fail(c, DSDTM_E_ARG, "dsdtm_batch_stage_keyframe: depth_scale must be > 0");
    const size_t B = c->prm.max_batch, K = DSDTM_TRACK_MAX_MATCHES, F = DSDTM_MAX_FEATS_LIMIT;
    if (!c->kf_circ_d) {
        // once per context at max_batch size: a captured step keeps pointing at these buffers
        if (dalloc(c, &c->kf_circ_d, B * 2 * K) || dalloc(c, &c->kf_ncirc_d, B) || dalloc(c, &c->kf_max_new_d, B) || dalloc(c, &c->kf_corner_d, B * F) ||
            dalloc(c, &c->kf_lifted_d, B * F) || dalloc(c, &c->kf_nnew_d, B) || dalloc(c, &c->kf_exact_d, B) || dalloc(c, &c->kf_depth_slot_d, B) ||
            dalloc(c, &c->kf_want_d, B) || dalloc(c, &c->kf_rows_d, B))
            return DSDTM_E_NOMEM;
    }
    std::vector<int32_t> rows;
    for (int i = 0; i < n; ++i) if (wt[i]) rows.push_back(i);
    cudaStream_t s = c->stream;
    DSDTM_CUDA(c, cudaMemcpyAsync(c->kf_depth_slot_d, ds.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->kf_want_d, wt.data(), n, cudaMemcpyHostToDevice, s));
    if (!rows.empty()) DSDTM_CUDA(c, cudaMemcpyAsync(c->kf_rows_d, rows.data(), rows.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    b.kf_staged = true; b.kf_min_dist = min_dist; b.kf_max_fts = max_fts; b.kf_thr = detection_threshold; b.kf_n_wanted = (int)rows.size();
    b.kf_want = wt; b.kf_depth_h = ds; b.commit_flags = 0; b.advance_flags = 0;
    for (int k = 0; k < 5; ++k) b.kf_dist[k] = dist[k];
    b.kf_depth_scale = any_depth ? depth_scale : 1.0f;
    drop_graphs(c);
    return 0;
}

// Tracking::CraeteKeyframe behind the tracked pose (dsdtm_batch_run bit 3): occupancy + circles -> FAST on the cur slots -> the sort and
// mask-circle selection -> the lift of the new corners, on the buffers of dsdtm_batch_stage_keyframe
static int enqueue_keyframe(dsdtm_ctx* c, cudaStream_t s, bool timed)
{
    auto& b = c->batch;
    if (timed) stage_begin(c, DSDTM_STAGE_FAST);
    DSDTM_CUDA(c, launch_keyframe_seed(c, b.n_pairs, b.kf_min_dist, b.kf_max_fts, s));
    DSDTM_CUDA(c, launch_fast_cells_slots(c, c->cur_slots_d, c->kf_rows_d, b.kf_n_wanted, b.kf_thr, s));
    DSDTM_CUDA(c, launch_detect_select(c, b.n_pairs, b.kf_thr, nullptr, c->kf_circ_d, 2 * DSDTM_TRACK_MAX_MATCHES, c->kf_ncirc_d, c->kf_max_new_d,
                                       c->kf_corner_d, b.kf_max_fts, c->kf_nnew_d, c->kf_exact_d, s));
    if (timed) stage_end(c, b.kf_n_wanted ? 3 : 2);
    if (timed) stage_begin(c, DSDTM_STAGE_INGEST);
    DSDTM_CUDA(c, launch_keyframe_lift_batch(c, b.n_pairs, b.kf_max_fts, b.kf_dist, b.kf_depth_scale, s));
    if (timed) stage_end(c, 1);
    return 0;
}

// SearchLocalPoints' selection + PoseOptimization behind the chain (dsdtm_batch_run bit 2), on the buffers of dsdtm_batch_stage_track
static int enqueue_track(dsdtm_ctx* c, cudaStream_t s, bool timed)
{
    auto& b = c->batch;
    const int ppp = b.store_staged ? b.store_cpf : b.map_ppp;
    if (timed) stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
    if (b.store_staged && b.store_found_live) DSDTM_CUDA(c, launch_track_select_store(c, b.n_pairs, b.store_cpf, c->st_found_d, (int)c->st_pts_n, s));
    else if (b.store_staged) DSDTM_CUDA(c, launch_track_select_store(c, b.n_pairs, b.store_cpf, c->sb_found_d, b.store_n_found, s));
    else DSDTM_CUDA(c, launch_track_select(c, b.n_pairs, b.feat_stride, b.map_ppp, s));
    if (timed) stage_end(c, 1);
    const PoseOptIo io = { c->trk_obs_d, c->trk_nobs_d, c->trk_pose_in_d, c->trk_pose_out_d, c->trk_res_d, c->trk_sum_d };
    if (timed) stage_begin(c, DSDTM_STAGE_POSE_OPT);
    DSDTM_CUDA(c, launch_pose_opt_io(c, io, b.n_pairs, DSDTM_TRACK_MAX_MATCHES, std::min(DSDTM_TRACK_MAX_MATCHES, ppp), b.track_iters, s));
    if (timed) stage_end(c, 1);
    return 0;
}

// the refinement chain of pairs [p0, p0 + n) on stream s: candidates from the aligned pose -> affine + search level -> warp -> Align2D -> records
static cudaError_t enqueue_chain(dsdtm_ctx* c, int p0, int n, int feat_stride, int ppp, int max_search_level, int align_iters, cudaStream_t s)
{
    cudaError_t e = launch_pair_candidates(c, p0, n, feat_stride, ppp, s);
    if (e == cudaSuccess) e = launch_candidate_prep(c, n * ppp, 0, max_search_level, s, p0 * ppp, c->cur_slots_d, ppp);
    if (e == cudaSuccess) e = launch_warp_affine(c, n * ppp, c->patches_d, s, p0 * ppp);
    if (e == cudaSuccess) e = launch_align2d(c, n * ppp, align_iters, s, p0 * ppp);
    if (e == cudaSuccess) e = launch_local_map_finalize(c, n * ppp, s, c->pair_reproj_d, p0 * ppp);
    return e;
}

// the kernels of one step, enqueued on stream s (captured into a CUDA graph by dsdtm_batch_run)
static int enqueue_step(dsdtm_ctx* c, int flags, cudaStream_t s, bool timed)
{
    auto& b = c->batch;
    const bool chain = (flags & 2) != 0;
    const int chunks = (timed || chain || c->step_chunks <= 1 || b.n_pairs < 4 * c->sm_count) ? 1 : std::min(c->step_chunks, kMaxStepStreams);
    if (chunks == 1) {
        if (flags & 1) {
            if (timed) stage_begin(c, DSDTM_STAGE_PYRAMID);
            DSDTM_CUDA(c, launch_pyramid_slots(c, c->cur_slots_d, b.n_pairs, s));
            if (timed) stage_end(c, pyramid_launches(c));
        }
        if (timed) stage_begin(c, DSDTM_STAGE_SPARSE_ALIGN);
        DSDTM_CUDA(c, launch_sparse_align(c, b.n_pairs, b.feat_stride, b.max_level, b.min_level, b.max_iters, false, s));
        if (timed) stage_end(c, 1);
        if (chain && b.store_staged) {
            // TrackWithLocalMap right after Run on the map store: per frame UpdateLocalMap over its key-frame rows, then the candidates
            const int n = b.n_pairs * b.store_cpf;
            if (timed) stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
            DSDTM_CUDA(c, launch_store_batch(c, b.n_pairs, b.store_all_rows, b.store_all_rows ? (int)c->st_kfs_n : b.store_range_max,
                                             b.store_max_local, b.store_cpf, b.max_search_level, s));
            if (timed) stage_end(c, 2);
            if (timed) stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
            DSDTM_CUDA(c, launch_warp_affine(c, n, c->patches_d, s));
            if (timed) stage_end(c, 1);
            if (timed) stage_begin(c, DSDTM_STAGE_ALIGN2D);
            DSDTM_CUDA(c, launch_align2d(c, n, b.map_align_iters, s, 0, nullptr, c->sb_rec_d));
            if (timed) stage_end(c, 1);
            if (flags & 4) {
                int r = enqueue_track(c, s, timed);
                if (r) return r;
            }
            if (flags & 8) {
                int r = enqueue_keyframe(c, s, timed);
                if (r) return r;
            }
        } else if (chain) {
            // TrackWithLocalMap right after Run: the patches come from the reference frame through the aligned pose, nothing from the host
            if (timed) stage_begin(c, DSDTM_STAGE_LOCAL_MAP);
            DSDTM_CUDA(c, launch_pair_candidates(c, 0, b.n_pairs, b.feat_stride, b.map_ppp, s));
            DSDTM_CUDA(c, launch_candidate_prep(c, b.n_pairs * b.map_ppp, 0, b.max_search_level, s, 0, c->cur_slots_d, b.map_ppp));
            if (timed) stage_end(c, 2);
            if (timed) stage_begin(c, DSDTM_STAGE_WARP_AFFINE);
            DSDTM_CUDA(c, launch_warp_affine(c, b.n_pairs * b.map_ppp, c->patches_d, s));
            if (timed) stage_end(c, 1);
            if (timed) stage_begin(c, DSDTM_STAGE_ALIGN2D);
            DSDTM_CUDA(c, launch_align2d(c, b.n_pairs * b.map_ppp, b.map_align_iters, s));
            DSDTM_CUDA(c, launch_local_map_finalize(c, b.n_pairs * b.map_ppp, s, c->pair_reproj_d, 0));
            if (timed) stage_end(c, 2);
            if (flags & 4) {
                int r = enqueue_track(c, s, timed);
                if (r) return r;
            }
            if (flags & 8) {
                int r = enqueue_keyframe(c, s, timed);
                if (r) return r;
            }
        } else if (b.patches_per_pair > 0) {
            if (timed) stage_begin(c, DSDTM_STAGE_ALIGN2D);
            DSDTM_CUDA(c, launch_align2d(c, b.n_pairs * b.patches_per_pair, b.align_iters, s));
            if (timed) stage_end(c, 1);
        }
        return 0;
    }
    // Chunked step: ALL pyramids are built on the origin stream first (a pair's ref slot may be the cur slot of a pair in another
    // chunk -- chained batches, ref[i] == cur[i-1] -- and its levels >= 1 must be complete before any alignment reads them, exactly
    // as in the unchunked order); then the pairs are split into `chunks` groups, each running sparse align -> Align2D on its own
    // stream (fork / join through events, captured into the same CUDA graph): the issue-bound Align2D kernel of one chunk fills the
    // idle issue slots of the latency-bound sparse-alignment kernel of another.
    const int per = (b.n_pairs + chunks - 1) / chunks;
    if (flags & 1) DSDTM_CUDA(c, launch_pyramid_slots(c, c->cur_slots_d, b.n_pairs, s));
    DSDTM_CUDA(c, cudaEventRecord(c->ev_fork, s));
    for (int k = 0; k < chunks; ++k) {
        const int p0 = k * per, n = std::min(per, b.n_pairs - p0);
        if (n <= 0) break;
        cudaStream_t sk = c->step_stream[k];
        DSDTM_CUDA(c, cudaStreamWaitEvent(sk, c->ev_fork, 0));
        DSDTM_CUDA(c, launch_sparse_align(c, n, b.feat_stride, b.max_level, b.min_level, b.max_iters, false, sk, p0, b.n_pairs));
        if (b.patches_per_pair > 0) DSDTM_CUDA(c, launch_align2d(c, n * b.patches_per_pair, b.align_iters, sk, p0 * b.patches_per_pair));
        DSDTM_CUDA(c, cudaEventRecord(c->ev_join[k], sk));
        DSDTM_CUDA(c, cudaStreamWaitEvent(s, c->ev_join[k], 0));
    }
    return 0;
}

int dsdtm_batch_run(dsdtm_ctx* c, int flags)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: no staged batch");
    if ((flags & 2) && !(b.map_staged || b.store_staged))
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: flags bit 1 needs dsdtm_batch_stage_map or dsdtm_batch_stage_store");
    if ((flags & 2) && b.store_staged) {
        // the store may have changed since staging (every change dropped the captured steps): the ranges and the prelude must still fit
        if (c->st_kfs_n == 0 || (size_t)b.store_range_end > c->st_kfs_n)
            return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: the map store no longer holds the staged key-frame ranges");
        if (check_store_batch_smem(c, b.store_all_rows ? (int)c->st_kfs_n : b.store_range_max, b.store_max_local, "dsdtm_batch_run"))
            return DSDTM_E_ARG;
    }
    if ((flags & 4) && !(flags & 2)) return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: flags bit 2 needs bit 1 (the refinement chain)");
    if ((flags & 4) && !b.track_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: flags bit 2 needs dsdtm_batch_stage_track");
    if ((flags & 8) && !(flags & 4)) return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: flags bit 3 needs bit 2 (the tracked pose)");
    if ((flags & 8) && !b.kf_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_run: flags bit 3 needs dsdtm_batch_stage_keyframe");
    const int gi = flags & 15;
    b.commit_flags = 0; b.advance_flags = 0;
    DSDTM_CUDA(c, cudaEventRecord(c->ev_a, c->stream));
    if (c->profiling) {
        // per-stage events cannot be recorded inside a captured graph: launch directly
        int r = enqueue_step(c, flags, c->stream, true);
        if (r) return r;
    } else {
        const int key[8] = { b.n_pairs, b.feat_stride, b.max_level, b.min_level, b.max_iters, b.patches_per_pair, b.align_iters, flags };
        if (!b.graph[gi] || std::memcmp(key, b.graph_key[gi], sizeof key) != 0) {
            if (b.graph[gi]) { cudaGraphExecDestroy(b.graph[gi]); b.graph[gi] = nullptr; }
            cudaGraph_t g = nullptr;
            const long long l0 = c->launches;
            DSDTM_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
            int r = enqueue_step(c, flags, c->stream, false);
            cudaError_t e = cudaStreamEndCapture(c->stream, &g);
            c->launches = l0;   // capture does not launch
            if (r) { if (g) cudaGraphDestroy(g); return r; }
            if (e != cudaSuccess) return fail(c, DSDTM_E_CUDA, "cudaStreamEndCapture", e);
            e = cudaGraphInstantiate(&b.graph[gi], g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) return fail(c, DSDTM_E_CUDA, "cudaGraphInstantiate", e);
            std::memcpy(b.graph_key[gi], key, sizeof key);
            ++c->captures;
            // re-record the start event after the (untimed) capture work
            DSDTM_CUDA(c, cudaEventRecord(c->ev_a, c->stream));
        }
        DSDTM_CUDA(c, cudaGraphLaunch(b.graph[gi], c->stream));
        {
            // what enqueue_step launched when the graph was captured (the capture's own tally was rolled back)
            const int chunks = (c->step_chunks <= 1 || b.n_pairs < 4 * c->sm_count) ? 1 : std::min(c->step_chunks, kMaxStepStreams);
            const int pyr = (flags & 1) ? pyramid_launches(c) : 0;
            if (flags & 2) c->launches += pyr + 1 + (b.store_staged ? 4 : 5) + ((flags & 4) ? 2 : 0) + ((flags & 8) ? (b.kf_n_wanted ? 4 : 3) : 0);
            else c->launches += pyr + (long long)chunks * (1 + (b.patches_per_pair > 0 ? 1 : 0));
        }
    }
    DSDTM_CUDA(c, cudaEventRecord(c->ev_b, c->stream));
    b.commit_flags = (b.store_staged && (flags & 4)) ? flags : 0;   // what dsdtm_batch_commit_store may apply
    return 0;
}

int dsdtm_batch_fetch(dsdtm_ctx* c, double* poses_out, int* n_tracked, double* patch_px_out, uint8_t* patch_conv)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_fetch: no staged batch");
    cudaStream_t s = c->stream;
    if (poses_out) DSDTM_CUDA(c, cudaMemcpyAsync(poses_out, c->poses_out_d, (size_t)b.n_pairs * 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (n_tracked) DSDTM_CUDA(c, cudaMemcpyAsync(n_tracked, c->n_tracked_d, (size_t)b.n_pairs * sizeof(int), cudaMemcpyDeviceToHost, s));
    const size_t np = (size_t)b.n_pairs * b.patches_per_pair;
    if (np && patch_px_out) DSDTM_CUDA(c, cudaMemcpyAsync(patch_px_out, c->patch_px_d, np * 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (np && patch_conv) DSDTM_CUDA(c, cudaMemcpyAsync(patch_conv, c->patch_conv_d, np, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->last_run_ms = ms;
    return 0;
}

int dsdtm_batch_fetch_map(dsdtm_ctx* c, dsdtm_reproj* reproj_out)
{
    if (!c || !reproj_out) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !b.map_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_fetch_map: no staged map batch");
    DSDTM_CUDA(c, cudaMemcpyAsync(reproj_out, c->pair_reproj_d, (size_t)b.n_pairs * b.map_ppp * sizeof(dsdtm_reproj), cudaMemcpyDeviceToHost, c->stream));
    DSDTM_CUDA(c, cudaStreamSynchronize(c->stream));
    return 0;
}

int dsdtm_batch_fetch_track(dsdtm_ctx* c, double* poses_c2w_out, int32_t* n_matches, dsdtm_match* matches, double* res_norm,
                            dsdtm_ba_summary* summaries)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !(b.map_staged || b.store_staged) || !b.track_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_fetch_track: no staged track batch");
    cudaStream_t s = c->stream;
    const size_t n = (size_t)b.n_pairs, K = DSDTM_TRACK_MAX_MATCHES;
    if (poses_c2w_out) DSDTM_CUDA(c, cudaMemcpyAsync(poses_c2w_out, c->trk_pose_out_d, n * 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (n_matches) DSDTM_CUDA(c, cudaMemcpyAsync(n_matches, c->trk_nobs_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (matches) DSDTM_CUDA(c, cudaMemcpyAsync(matches, c->trk_match_d, n * K * sizeof(dsdtm_match), cudaMemcpyDeviceToHost, s));
    if (res_norm) DSDTM_CUDA(c, cudaMemcpyAsync(res_norm, c->trk_res_d, n * K * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (summaries) DSDTM_CUDA(c, cudaMemcpyAsync(summaries, c->trk_sum_d, n * sizeof(dsdtm_ba_summary), cudaMemcpyDeviceToHost, s));
    std::vector<int32_t> nm;
    std::vector<double> prior;
    if (b.store_staged) {
        // match counts change with the store between replays, and an overflowed frame (-1) keeps its prior pose
        nm.resize(n); prior.resize(n * 7);
        DSDTM_CUDA(c, cudaMemcpyAsync(nm.data(), c->trk_nobs_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
        DSDTM_CUDA(c, cudaMemcpyAsync(prior.data(), c->trk_pose_in_d, n * 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    for (size_t i = 0; i < nm.size(); ++i) {
        const size_t k = (size_t)std::max(nm[i], 0);
        if (matches) std::memset(matches + i * K + k, 0, (K - k) * sizeof(dsdtm_match));
        if (res_norm) std::memset(res_norm + i * K + k, 0, (K - k) * sizeof(double));
        if (nm[i] < 0 && poses_c2w_out) std::memcpy(poses_c2w_out + 7 * i, prior.data() + 7 * i, 7 * sizeof(double));
    }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->last_run_ms = ms;
    return 0;
}

int dsdtm_batch_fetch_keyframe(dsdtm_ctx* c, int32_t* n_new, dsdtm_corner* corners, dsdtm_lifted* lifted, uint8_t* exact_path)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !(b.map_staged || b.store_staged) || !b.track_staged || !b.kf_staged)
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_fetch_keyframe: no staged key-frame batch");
    cudaStream_t s = c->stream;
    const size_t n = (size_t)b.n_pairs, F = (size_t)b.kf_max_fts;
    std::vector<int32_t> nn(n);
    DSDTM_CUDA(c, cudaMemcpyAsync(nn.data(), c->kf_nnew_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (corners) DSDTM_CUDA(c, cudaMemcpyAsync(corners, c->kf_corner_d, n * F * sizeof(dsdtm_corner), cudaMemcpyDeviceToHost, s));
    if (lifted) DSDTM_CUDA(c, cudaMemcpyAsync(lifted, c->kf_lifted_d, n * F * sizeof(dsdtm_lifted), cudaMemcpyDeviceToHost, s));
    if (exact_path) DSDTM_CUDA(c, cudaMemcpyAsync(exact_path, c->kf_exact_d, n, cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    // the step writes rows < n_new[i] only: what lies past them is left from earlier replays and is cleared here
    for (size_t i = 0; i < n; ++i) {
        const size_t k = (size_t)std::max(nn[i], 0);
        if (corners) std::memset(corners + i * F + k, 0, (F - k) * sizeof(dsdtm_corner));
        if (lifted) std::memset(lifted + i * F + k, 0, (F - k) * sizeof(dsdtm_lifted));
    }
    if (n_new) std::memcpy(n_new, nn.data(), n * sizeof(int32_t));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->last_run_ms = ms;
    return 0;
}

int dsdtm_batch_commit_store(dsdtm_ctx* c, float outlier_threshold, const int32_t* kf_rows, int32_t* kf_row_out, int32_t* point_first_out,
                             int32_t* n_points_out)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !b.store_staged || !b.track_staged || !b.commit_flags)
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_commit_store: no store-mode run with flags bit 2 since the last staging or commit");
    if (std::isnan(outlier_threshold)) return fail(c, DSDTM_E_ARG, "dsdtm_batch_commit_store: outlier_threshold is NaN");
    const int n = b.n_pairs;
    const bool kf = (b.commit_flags & 8) != 0 && b.kf_staged;
    int n_w = 0;
    if (kf) for (int i = 0; i < n; ++i) n_w += b.kf_want[(size_t)i] ? 1 : 0;
    if (kf && kf_rows) {
        // every wanted frame names its own empty key frame (dsdtm_store_append_keyframe with no features)
        std::vector<uint8_t> named(c->st_kfs_n, 0);
        for (int i = 0; i < n; ++i) {
            if (!b.kf_want[(size_t)i]) continue;
            const int r = kf_rows[i];
            if (r < 0 || (size_t)r >= c->st_kfs_n) return fail(c, DSDTM_E_ARG, "dsdtm_batch_commit_store: reserved key-frame row outside the table");
            if (c->st_kf_nfeat[(size_t)r] != 0) return fail(c, DSDTM_E_ARG, "dsdtm_batch_commit_store: reserved key-frame row is not empty");
            if (named[(size_t)r]) return fail(c, DSDTM_E_ARG, "dsdtm_batch_commit_store: two frames name the same key-frame row");
            named[(size_t)r] = 1;
        }
    }
    // the worst case, reserved before anything is enqueued: every wanted frame a key frame of max(Max_fts, 200) features, all new corners
    // with a point
    const size_t F0 = c->st_feats_n, P0 = c->st_pts_n, K0 = c->st_kfs_n;
    const size_t max_f = (size_t)n_w * (size_t)std::max(b.kf_max_fts, DSDTM_TRACK_MAX_MATCHES), max_p = (size_t)n_w * (size_t)b.kf_max_fts;
    const size_t max_k = kf_rows ? 0 : (size_t)n_w;
    if (F0 + max_f > (size_t)INT32_MAX || P0 + max_p > (size_t)INT32_MAX) return fail(c, DSDTM_E_ARG, "dsdtm_batch_commit_store: tables beyond 32-bit rows");
    const size_t old_claim_cap = c->st_claim_cap;
    // what a captured store-mode step points at: a commit that moves none of these tables and writes no key frame keeps the captures
    const void* tables0[] = { c->st_feats_d, c->st_pts_d, c->st_found_d, c->st_claim_d, c->st_kfs_d, c->st_vis_d, c->st_dist_d };
    if (grow_keep(c, &c->st_feats_d, &c->st_feats_cap, F0 + max_f, F0) || grow_keep(c, &c->st_pts_d, &c->st_pts_cap, P0 + max_p, P0) ||
        grow_keep(c, &c->st_found_d, &c->st_found_cap, P0 + max_p, P0) || grow_keep(c, &c->st_claim_d, &c->st_claim_cap, P0 + max_p, P0) ||
        grow_keep(c, &c->st_kfs_d, &c->st_kfs_cap, K0 + max_k, K0) || grow(c, &c->st_vis_d, &c->st_vis_cap, K0 + max_k) ||
        grow(c, &c->st_dist_d, &c->st_dist_cap, K0 + max_k) || grow(c, &c->cm_d, &c->cm_cap, (size_t)9 * n + 4) ||
        grow(c, &c->cm_push_d, &c->cm_push_cap, std::max(max_f, (size_t)1)))
        return DSDTM_E_NOMEM;
    if (!c->st_sel_d && dalloc(c, &c->st_sel_d, 32)) return DSDTM_E_NOMEM;
    if (ensure_pinned(c, ((size_t)6 * n + 4) * sizeof(int32_t))) return DSDTM_E_NOMEM;
    c->st_kf_nfeat.reserve(K0 + max_k);
    c->st_kf_slot.reserve(K0 + max_k);
    const void* tables1[] = { c->st_feats_d, c->st_pts_d, c->st_found_d, c->st_claim_d, c->st_kfs_d, c->st_vis_d, c->st_dist_d };
    if (std::memcmp(tables0, tables1, sizeof tables0) != 0) drop_store_graphs(c);
    cudaStream_t s = c->stream;
    if (c->st_claim_cap != old_claim_cap)     // fresh part of the claim array: "never claimed" (as dsdtm_store_set_points)
        DSDTM_CUDA(c, cudaMemsetAsync(c->st_claim_d + P0, 0xFF, (c->st_claim_cap - P0) * sizeof(unsigned long long), s));
    int* rows_d = c->cm_d + 8 * (size_t)n + 4;
    if (kf && kf_rows) DSDTM_CUDA(c, cudaMemcpyAsync(rows_d, kf_rows, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    StoreCommitArgs a;
    a.threshold = outlier_threshold; a.keyframes = kf; a.kf_rows_d = (kf && kf_rows) ? rows_d : nullptr;
    a.cnt_d = c->cm_d; a.out_d = c->cm_d + 3 * (size_t)n; a.push_d = c->cm_push_d;
    DSDTM_CUDA(c, launch_store_commit(c, a, s));
    const int committed = b.commit_flags;
    b.commit_flags = 0; b.advance_flags = 0;                       // enqueued: a second commit of this run is a state error whatever happens below
    int32_t* out_h = reinterpret_cast<int32_t*>(c->pinned);
    DSDTM_CUDA(c, cudaMemcpyAsync(out_h, a.out_d, ((size_t)5 * n + 4) * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    int32_t* nm_h = out_h + 5 * (size_t)n + 4;                // the match counts, for dsdtm_batch_advance's held frames
    DSDTM_CUDA(c, cudaMemcpyAsync(nm_h, c->trk_nobs_d, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    const int32_t* tot = out_h + 5 * (size_t)n;
    if (tot[2] != 0) drop_store_graphs(c);    // a key frame: new rows, a reserved row filled, maybe a wider st_max_feats
    c->st_feats_n = F0 + (size_t)tot[0];
    c->st_pts_n = P0 + (size_t)tot[1];
    if (!kf_rows) c->st_kfs_n = K0 + (size_t)tot[2];
    c->st_kf_nfeat.resize(c->st_kfs_n, 0);
    c->st_kf_slot.resize(c->st_kfs_n, 0);
    for (int i = 0; i < n; ++i)
        if (out_h[i] >= 0) {
            c->st_kf_nfeat[(size_t)out_h[i]] = out_h[4 * (size_t)n + i];
            c->st_kf_slot[(size_t)out_h[i]] = b.cur_h[(size_t)i];
        }
    c->st_max_feats = std::max(c->st_max_feats, (int)tot[3]);
    b.nm_h.assign(nm_h, nm_h + n);
    b.advance_flags = committed;
    if (kf_row_out) std::memcpy(kf_row_out, out_h, (size_t)n * sizeof(int32_t));
    if (point_first_out) std::memcpy(point_first_out, out_h + n, (size_t)n * sizeof(int32_t));
    if (n_points_out) std::memcpy(n_points_out, out_h + 2 * (size_t)n, (size_t)n * sizeof(int32_t));
    return 0;
}

int dsdtm_batch_advance(dsdtm_ctx* c, const int32_t* next_cur_slots, const uint8_t* hold, const uint8_t* want_next, uint8_t* status_out)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged || !b.store_staged || !b.track_staged || !b.advance_flags)
        return fail(c, DSDTM_E_STATE, "dsdtm_batch_advance: no committed store-mode run with flags 7 or 15 since the last staging or advance");
    if (want_next && !b.kf_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_advance: want_next needs dsdtm_batch_stage_keyframe");
    if (!next_cur_slots) return fail(c, DSDTM_E_ARG, "dsdtm_batch_advance: next_cur_slots is NULL");
    const int n = b.n_pairs;
    const bool kf = (b.advance_flags & 8) != 0 && b.kf_staged;
    if (b.feat_stride < std::max(DSDTM_TRACK_MAX_MATCHES, b.kf_staged ? b.kf_max_fts : 0))
        return fail(c, DSDTM_E_ARG, "dsdtm_batch_advance: feat_stride below max(DSDTM_TRACK_MAX_MATCHES, max_fts): a frame's features would not fit");
    // the decisions, on the host: which frames advance (as key frames), and their reference slots afterwards
    std::vector<int32_t> adv((size_t)2 * n);
    std::vector<int32_t> ref_next(b.ref_h);
    for (int i = 0; i < n; ++i) {
        const int mode = b.nm_h[(size_t)i] < 0 ? DSDTM_ADV_HELD_OVERFLOW : (hold && hold[i]) ? DSDTM_ADV_HELD_CALLER
                       : (kf && b.kf_want[(size_t)i]) ? DSDTM_ADV_KEYFRAME : DSDTM_ADV_ADVANCED;
        adv[(size_t)i] = next_cur_slots[i];
        adv[(size_t)n + i] = mode;
        if (mode <= DSDTM_ADV_KEYFRAME) ref_next[(size_t)i] = b.cur_h[(size_t)i];
    }
    std::vector<uint8_t> named((size_t)c->prm.max_frames, 0);
    // a key frame's pyramid must stay; an empty reserved row (no features: never close, never local) reads no slot and is skipped
    for (size_t r = 0; r < c->st_kf_slot.size(); ++r) {
        const int32_t sl = c->st_kf_slot[r];
        if (c->st_kf_nfeat[r] != 0 && sl >= 0 && sl < c->prm.max_frames) named[(size_t)sl] = 1;
    }
    for (int32_t s : ref_next) named[(size_t)s] |= 2;
    for (int i = 0; i < n; ++i) {
        const int s = next_cur_slots[i];
        if (s < 0 || s >= c->prm.max_frames) return fail(c, DSDTM_E_ARG, "dsdtm_batch_advance: next cur slot out of range");
        if (named[(size_t)s] & 1) return fail(c, DSDTM_E_ARG, "dsdtm_batch_advance: next cur slot holds a key frame of the store");
        if (named[(size_t)s] & 2) return fail(c, DSDTM_E_ARG, "dsdtm_batch_advance: next cur slot is a reference slot after the advance");
        if (named[(size_t)s] & 4) return fail(c, DSDTM_E_ARG, "dsdtm_batch_advance: next cur slot named twice");
        named[(size_t)s] |= 4;
    }
    std::vector<uint8_t> wt;
    std::vector<int32_t> rows;
    if (want_next) {
        wt.resize((size_t)n);
        for (int i = 0; i < n; ++i) if ((wt[(size_t)i] = want_next[i] ? 1 : 0)) rows.push_back(i);
    }
    if (!c->adv_d && dalloc(c, &c->adv_d, (size_t)2 * c->prm.max_batch)) return DSDTM_E_NOMEM;
    if (ensure_pinned(c, adv.size() * sizeof(int32_t) + 2 * (size_t)n * sizeof(int32_t))) return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    int32_t* pin = reinterpret_cast<int32_t*>(c->pinned);
    std::memcpy(pin, adv.data(), adv.size() * sizeof(int32_t));
    DSDTM_CUDA(c, cudaMemcpyAsync(c->adv_d, pin, adv.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    DSDTM_CUDA(c, launch_sequence_advance(c, c->adv_d, kf, s));
    // enqueued: the host mirrors follow the device from here, and a second advance of this commit is a state error whatever happens below
    b.advance_flags = 0;
    for (int i = 0; i < n; ++i) b.cur_h[(size_t)i] = next_cur_slots[i];
    b.ref_h = ref_next;
    if (want_next) {
        // after the advance, so that a launch that fails leaves the want mask as it was on the device and on the host alike
        int32_t* rp = pin + adv.size();
        uint8_t* wp = reinterpret_cast<uint8_t*>(rp + n);
        if (!rows.empty()) std::memcpy(rp, rows.data(), rows.size() * sizeof(int32_t));
        std::memcpy(wp, wt.data(), (size_t)n);
        DSDTM_CUDA(c, cudaMemcpyAsync(c->kf_want_d, wp, (size_t)n, cudaMemcpyHostToDevice, s));
        if (!rows.empty()) DSDTM_CUDA(c, cudaMemcpyAsync(c->kf_rows_d, rp, rows.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        // the wanted count sizes the FAST grid of the captured flags-8 steps; the mask and the rows are read from device memory
        if ((int)rows.size() != b.kf_n_wanted)
            for (int gi = 8; gi < 16; ++gi)
                if (b.graph[gi]) { cudaGraphExecDestroy(b.graph[gi]); b.graph[gi] = nullptr; }
        b.kf_want = wt; b.kf_n_wanted = (int)rows.size();
    }
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    if (status_out)
        for (int i = 0; i < n; ++i) status_out[i] = (uint8_t)adv[(size_t)n + i];
    return 0;
}

int dsdtm_batch_upload_step(dsdtm_ctx* c, const uint8_t* imgs, const uint16_t* depth)
{
    if (!c || !imgs) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_upload_step: no staged batch");
    if (depth && !b.kf_staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_upload_step: depth needs dsdtm_batch_stage_keyframe's depth slots");
    const int n = b.n_pairs;
    const size_t px = (size_t)c->cam.width * c->cam.height;
    if (depth && ensure_depth_pool(c)) return DSDTM_E_NOMEM;
    cudaStream_t s = c->stream;
    bool contiguous = true;
    for (int i = 1; i < n; ++i) contiguous &= b.cur_h[(size_t)i] == b.cur_h[0] + i;
    // level 0 of a slot is dense at offset 0 (stride == width)
    if (contiguous)
        DSDTM_CUDA(c, cudaMemcpy2DAsync(c->frames_d + (size_t)b.cur_h[0] * c->geo.frame_stride, c->geo.frame_stride, imgs, px, px, (size_t)n,
                                        cudaMemcpyHostToDevice, s));
    else
        for (int i = 0; i < n; ++i)
            DSDTM_CUDA(c, cudaMemcpyAsync(c->frames_d + (size_t)b.cur_h[(size_t)i] * c->geo.frame_stride, imgs + (size_t)i * px, px,
                                          cudaMemcpyHostToDevice, s));
    if (depth)
        for (int i = 0; i < n; ++i) {
            const int ds = b.kf_depth_h[(size_t)i];
            if (ds >= 0)
                DSDTM_CUDA(c, cudaMemcpyAsync(c->depth_d + (size_t)ds * px, depth + (size_t)i * px, px * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
        }
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

int dsdtm_batch_fetch_ref(dsdtm_ctx* c, int32_t* ref_slots, int32_t* cur_slots, dsdtm_ref_feat* feats, int32_t* n_feats, double* centers,
                          double* poses_ref, double* poses_in)
{
    if (!c) return DSDTM_E_ARG;
    auto& b = c->batch;
    if (!b.staged) return fail(c, DSDTM_E_STATE, "dsdtm_batch_fetch_ref: no staged batch");
    const size_t n = (size_t)b.n_pairs;
    cudaStream_t s = c->stream;
    if (ref_slots) DSDTM_CUDA(c, cudaMemcpyAsync(ref_slots, c->ref_slots_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (cur_slots) DSDTM_CUDA(c, cudaMemcpyAsync(cur_slots, c->cur_slots_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (feats) DSDTM_CUDA(c, cudaMemcpyAsync(feats, c->feats_d, n * b.feat_stride * sizeof(dsdtm_ref_feat), cudaMemcpyDeviceToHost, s));
    if (n_feats) DSDTM_CUDA(c, cudaMemcpyAsync(n_feats, c->n_feats_d, n * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    if (centers) DSDTM_CUDA(c, cudaMemcpyAsync(centers, c->centers_d, n * 3 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (poses_ref) DSDTM_CUDA(c, cudaMemcpyAsync(poses_ref, c->poses_ref_d, n * 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (poses_in) DSDTM_CUDA(c, cudaMemcpyAsync(poses_in, c->poses_in_d, n * 7 * sizeof(double), cudaMemcpyDeviceToHost, s));
    DSDTM_CUDA(c, cudaStreamSynchronize(s));
    return 0;
}

float dsdtm_last_run_ms(const dsdtm_ctx* c) { return c ? c->last_run_ms : 0.f; }

int dsdtm_timer_start(dsdtm_ctx* c)
{
    if (!c) return DSDTM_E_ARG;
    DSDTM_CUDA(c, cudaEventRecord(c->ev_t0, c->stream));
    return 0;
}

float dsdtm_timer_stop(dsdtm_ctx* c)
{
    if (!c) return -1.f;
    float ms = -1.f;
    if (cudaEventRecord(c->ev_t1, c->stream) != cudaSuccess || cudaEventSynchronize(c->ev_t1) != cudaSuccess ||
        cudaEventElapsedTime(&ms, c->ev_t0, c->ev_t1) != cudaSuccess) {
        fail(c, DSDTM_E_CUDA, "dsdtm_timer_stop", cudaGetLastError());
        return -1.f;
    }
    return ms;
}

// chain != nullptr: the refinement inputs come from the reference frames on the device (dsdtm_track_batch_e2e) instead of host patches
struct E2eChain { const double* poses_ref; int ppp; int max_search_level; dsdtm_reproj* reproj_out; };

static int pair_batch_e2e_impl(dsdtm_ctx* c, int n_pairs, const uint8_t* cur_imgs, const int* ref_slots, const int* cur_slots,
                         const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats, const double* ref_centers,
                         const double* poses_in, int max_level, int min_level, int max_iters, const uint8_t* patches10,
                         const double* patch_px, const int* patch_level, int ppp, int align_iters, double* poses_out,
                         int* n_tracked, double* patch_px_out, uint8_t* patch_conv, const E2eChain* chain)
{
    if (!c || !cur_imgs || !ref_slots || !cur_slots || !feats || !n_feats || !ref_centers || !poses_in || !poses_out || !n_tracked) return DSDTM_E_ARG;
    if (check_grid_frames(c, n_pairs) || check_pairs(c, n_pairs, ref_slots, cur_slots, feat_stride, n_feats, max_level, min_level, max_iters))
        return DSDTM_E_ARG;
    if (ppp < 0 || ppp > c->prm.max_patches || align_iters < 0) return fail(c, DSDTM_E_ARG, "patches_per_pair > max_patches");
    if (ppp > 0 && (!patches10 || !patch_px || !patch_level || !patch_px_out || !patch_conv)) return fail(c, DSDTM_E_ARG, "null patch arrays");
    c->batch.staged = false; c->batch.commit_flags = 0; c->batch.advance_flags = 0;
    const LevelGeom& g = c->geo;
    const size_t img_bytes = (size_t)g.w[0] * g.h[0];
    // chunked pipeline: H2D of chunk k+1 (copy stream) overlaps the kernels of chunk k (compute stream) and the D2H of chunk k-1.
    // Precondition for the overlap: no pair reads, as its reference, a slot that this call uploads as ANOTHER pair's current frame
    // (chained batches, ref[i] == cur[i-1]); otherwise the upload / pyramid of one chunk would race the alignment of another.
    // Such batches run as ONE chunk: upload all, build all pyramids, then align -- the order of dsdtm_batch_run.
    bool chained = false;
    {
        std::vector<unsigned char> is_cur((size_t)c->prm.max_frames, 0);
        for (int i = 0; i < n_pairs; ++i) is_cur[(size_t)cur_slots[i]] = 1;
        for (int i = 0; i < n_pairs && !chained; ++i) chained = is_cur[(size_t)ref_slots[i]] != 0;
    }
    const int n_chunks = chained ? 1 : std::max(1, std::min(8, n_pairs / 64));
    const int per = (n_pairs + n_chunks - 1) / n_chunks;
    cudaStream_t cs = c->copy_stream[0], ds = c->copy_stream[1], ks = c->stream;
    int rc = 0;
    cudaError_t ce = cudaSuccess;
#define E2E_CK(call, what) do { if (!rc && (ce = (call)) != cudaSuccess) rc = fail(c, DSDTM_E_CUDA, what, ce); } while (0)
    DSDTM_CUDA(c, cudaEventRecord(c->ev_a, ks));
    DSDTM_CUDA(c, cudaStreamWaitEvent(cs, c->ev_a, 0));
    for (int k = 0; k < n_chunks && !rc; ++k) {
        const int p0 = k * per, n = std::min(per, n_pairs - p0);
        if (n <= 0) break;
        // cur images: scatter into their slots. Slots in arithmetic progression (the usual ref/cur interleaving gives
        // stride 2) collapse into ONE strided 2-D copy; per-image copies cost ~2x in DMA setup.
        int sstride = (n > 1) ? cur_slots[p0 + 1] - cur_slots[p0] : 1;
        bool regular = sstride > 0;
        for (int i = 1; i < n && regular; ++i) if (cur_slots[p0 + i] != cur_slots[p0] + i * sstride) regular = false;
        if (regular) {
            E2E_CK(cudaMemcpy2DAsync(c->frames_d + (size_t)cur_slots[p0] * g.frame_stride, (size_t)sstride * g.frame_stride,
                                     cur_imgs + (size_t)p0 * img_bytes, img_bytes, img_bytes, n, cudaMemcpyHostToDevice, cs), "H2D images");
        } else {
            for (int i = 0; i < n && !rc; ++i)
                E2E_CK(cudaMemcpyAsync(c->frames_d + (size_t)cur_slots[p0 + i] * g.frame_stride, cur_imgs + (size_t)(p0 + i) * img_bytes, img_bytes,
                                       cudaMemcpyHostToDevice, cs), "H2D image");
        }
        if (!rc) rc = stage_pairs(c, n, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_in, cs, p0);
        if (!rc) rc = stage_patches(c, n, cur_slots, patches10, patch_px, patch_level, ppp, cs, p0);
        if (chain) E2E_CK(cudaMemcpyAsync(c->poses_ref_d + 7 * (size_t)p0, chain->poses_ref + 7 * (size_t)p0, (size_t)n * 7 * sizeof(double), cudaMemcpyHostToDevice, cs), "H2D reference poses");
        E2E_CK(cudaEventRecord(c->ev_up[k], cs), "e2e event");
        E2E_CK(cudaStreamWaitEvent(ks, c->ev_up[k], 0), "e2e event");
        if (rc) break;
        if (ppp > 0) {
            fill_patch_slots_kernel<<<(n * ppp + 255) / 256, 256, 0, ks>>>(c->cur_slots_d, c->patch_slot_d, ppp, n * ppp, p0 * ppp);
            E2E_CK(cudaGetLastError(), "fill_patch_slots_kernel");
        }
        E2E_CK(launch_pyramid_slots(c, c->cur_slots_d + p0, n, ks), "e2e pyramid launch");
        E2E_CK(launch_sparse_align(c, n, feat_stride, max_level, min_level, max_iters, false, ks, p0, n_pairs), "e2e sparse-align launch");
        if (ppp > 0) E2E_CK(launch_align2d(c, n * ppp, align_iters, ks, p0 * ppp), "e2e align2d launch");
        if (chain) E2E_CK(enqueue_chain(c, p0, n, feat_stride, chain->ppp, chain->max_search_level, align_iters, ks), "e2e refinement chain launch");
        E2E_CK(cudaEventRecord(c->ev_done[k], ks), "e2e event");
        E2E_CK(cudaStreamWaitEvent(ds, c->ev_done[k], 0), "e2e event");
        E2E_CK(cudaMemcpyAsync(poses_out + 7 * (size_t)p0, c->poses_out_d + 7 * (size_t)p0, (size_t)n * 7 * sizeof(double), cudaMemcpyDeviceToHost, ds), "D2H poses");
        E2E_CK(cudaMemcpyAsync(n_tracked + p0, c->n_tracked_d + p0, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, ds), "D2H tracked counts");
        if (ppp > 0) {
            E2E_CK(cudaMemcpyAsync(patch_px_out + 2 * (size_t)p0 * ppp, c->patch_px_d + 2 * (size_t)p0 * ppp, (size_t)n * ppp * 2 * sizeof(double), cudaMemcpyDeviceToHost, ds), "D2H patch positions");
            E2E_CK(cudaMemcpyAsync(patch_conv + (size_t)p0 * ppp, c->patch_conv_d + (size_t)p0 * ppp, (size_t)n * ppp, cudaMemcpyDeviceToHost, ds), "D2H patch flags");
        }
        if (chain) E2E_CK(cudaMemcpyAsync(chain->reproj_out + (size_t)p0 * chain->ppp, c->pair_reproj_d + (size_t)p0 * chain->ppp,
                                          (size_t)n * chain->ppp * sizeof(dsdtm_reproj), cudaMemcpyDeviceToHost, ds), "D2H refinement records");
    }
#undef E2E_CK
    cudaEventRecord(c->ev_chunk[0], ds);
    cudaStreamWaitEvent(ks, c->ev_chunk[0], 0);
    cudaEventRecord(c->ev_b, ks);
    cudaError_t e = cudaStreamSynchronize(ks);
    const cudaError_t e2 = cudaStreamSynchronize(cs), e3 = cudaStreamSynchronize(ds);
    if (rc) return rc;
    if (e == cudaSuccess) e = (e2 != cudaSuccess) ? e2 : e3;
    if (e != cudaSuccess) return fail(c, DSDTM_E_CUDA, "e2e sync", e);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev_a, c->ev_b) == cudaSuccess) c->last_run_ms = ms;
    return 0;
}

int dsdtm_pair_batch_e2e(dsdtm_ctx* c, int n_pairs, const uint8_t* cur_imgs, const int* ref_slots, const int* cur_slots,
                         const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats, const double* ref_centers,
                         const double* poses_in, int max_level, int min_level, int max_iters, const uint8_t* patches10,
                         const double* patch_px, const int* patch_level, int ppp, int align_iters, double* poses_out,
                         int* n_tracked, double* patch_px_out, uint8_t* patch_conv)
{
    return pair_batch_e2e_impl(c, n_pairs, cur_imgs, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_in, max_level, min_level,
                               max_iters, patches10, patch_px, patch_level, ppp, align_iters, poses_out, n_tracked, patch_px_out, patch_conv, nullptr);
}

int dsdtm_track_batch_e2e(dsdtm_ctx* c, int n_pairs, const uint8_t* cur_imgs, const int* ref_slots, const int* cur_slots,
                          const dsdtm_ref_feat* feats, int feat_stride, const int* n_feats, const double* ref_centers,
                          const double* poses_ref_c2w, const double* poses_c2r_in, int max_level, int min_level, int max_iters,
                          int points_per_pair, int max_search_level, int align_iters, double* poses_c2r_out, int* n_tracked,
                          dsdtm_reproj* reproj_out)
{
    if (!c || !poses_ref_c2w || !reproj_out) return DSDTM_E_ARG;
    if (points_per_pair < 1 || points_per_pair > c->prm.max_patches || points_per_pair > feat_stride)
        return fail(c, DSDTM_E_ARG, "points_per_pair must be 1..min(max_patches, feat_stride)");
    if (max_search_level < 0 || max_search_level >= c->geo.levels) return fail(c, DSDTM_E_ARG, "bad max_search_level");
    const E2eChain ch = { poses_ref_c2w, points_per_pair, max_search_level, reproj_out };
    return pair_batch_e2e_impl(c, n_pairs, cur_imgs, ref_slots, cur_slots, feats, feat_stride, n_feats, ref_centers, poses_c2r_in, max_level, min_level,
                               max_iters, nullptr, nullptr, nullptr, 0, align_iters, poses_c2r_out, n_tracked, nullptr, nullptr, &ch);
}

}  // extern "C"
