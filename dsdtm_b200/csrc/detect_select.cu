// detect_select.cu -- the second half of Feature_detector::detect (ref: src/Feature_detection.cpp:111-150) on the cell keys that
// fast_kernel left in cells_d: score sort, mask test and filled circles, up to Max_fts - mvFeatures.size() additions.
//
//   detect_select_kernel : one CTA per frame.
//     1. decode : key -> corner exactly as capi.cu's decode_cells (empty cell = {0, 0, 0, seed}, x and y shifted by the level).
//     2. order  : the cells scoring above 20 are ranked by counting, key (score descending, cell index). If two of them tie, the
//                 order of equal scores is whatever libstdc++'s introsort makes of the whole cell array, so one thread re-sorts
//                 all n_cells decoded cells (cell order in, as the reference builds its vector) with std_sort.cuh. Without a tie
//                 every correct sort puts the cells above 20 first in one and the same order, and the rest never matter: the
//                 "> 20" filter skips them and only additions count toward the cap.
//     3. mask   : a shared-memory bitmap of the image, bit set = pixel != 255, seeded from the caller's mask image and prior
//                 circles. Circles are the clipped row spans of cv::circle(.., -1) (OpenCV's filled midpoint circle), the span
//                 table select.cu's track_select_kernel uses, built here for every radius 0..kMaxRadius.
//     4. walk   : warp 0 takes the candidates 32 at a time in that order; each lane tests its bit (the corner position is
//                 integral, so cvRound of the float position is the position), the first free lane wins, the warp paints its
//                 CellSize circle and the lanes behind the winner test again. Stops after max_new additions.
#include "ctx.cuh"
#include "std_sort.cuh"

namespace dsdtm {

namespace {

static const int kThreads = 512;
static const int kMaxRadius = 64;                 // also the bound on dsdtm_circle.radius
static const int kSpanPitch = kMaxRadius + 1;
static const float kMinScore = 20.f;              // ref: :128 literal
static const size_t kMaxBitmapBytes = 24 * 4 * 480;   // 752 x 480 pixels, rows padded to whole 32-bit words: 45 KB

struct DetSelArgs {
    const unsigned long long* cells; int n_cells; float seed;
    int w, h, pitch;                              // image, bitmap row pitch in 32-bit words
    int cell_size;
    const uint8_t* masks;                         // n * h * w or null
    const dsdtm_circle* circles; int circle_stride; const int* n_circles;   // circles / n_circles may be null
    const int* max_new;
    dsdtm_corner* out; int out_stride; int* n_out; uint8_t* exact;
};

struct Cand { float score; int cell; };           // the literal sort's element: only the score is compared

__device__ __forceinline__ dsdtm_corner decode(unsigned long long k, float seed)
{
    if (k == 0) return dsdtm_corner{ 0, 0, 0, seed };                                   // ref: :74
    const unsigned order = ~(unsigned)(k & 0xFFFFFFFFull);
    const int L = order >> 28, y = (order >> 14) & 0x3FFF, x = order & 0x3FFF;
    return dsdtm_corner{ x << L, y << L, L, __uint_as_float((unsigned)(k >> 32)) };     // ref: :106
}

// rows cy - r .. cy + r of the filled circle, clipped to the image; lanes (or threads) `t0, t0 + step, ..` take one row each
__device__ __forceinline__ void paint_rows(unsigned* bm, const DetSelArgs& a, const uint8_t* span, long long cx, long long cy, int r,
                                           int t0, int step, bool atomic)
{
    for (int dy = -r + t0; dy <= r; dy += step) {
        const long long y = cy + dy;
        if (y < 0 || y >= a.h) continue;
        const int s = span[r * kSpanPitch + (dy < 0 ? -dy : dy)];
        const long long x0l = cx - s < 0 ? 0 : cx - s, x1l = cx + s > a.w - 1 ? a.w - 1 : cx + s;
        if (x0l > x1l) continue;
        const int x0 = (int)x0l, x1 = (int)x1l;
        unsigned* row = bm + (size_t)y * a.pitch;
        for (int wd = x0 >> 5; wd <= (x1 >> 5); ++wd) {
            const int lo = max(x0 - 32 * wd, 0), hi = min(x1 - 32 * wd, 31);
            const unsigned m = (hi == 31 ? 0xFFFFFFFFu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
            if (atomic) atomicOr(row + wd, m);
            else row[wd] |= m;
        }
    }
}

__device__ __forceinline__ bool masked(const unsigned* bm, int pitch, int x, int y) { return (bm[(size_t)y * pitch + (x >> 5)] >> (x & 31)) & 1u; }

__global__ void __launch_bounds__(kThreads) detect_select_kernel(const DetSelArgs a)
{
    extern __shared__ __align__(16) unsigned char ds_smem[];
    __shared__ int s_m, s_tie;
    const int frame = blockIdx.x, tid = threadIdx.x;
    unsigned* bm = reinterpret_cast<unsigned*>(ds_smem);
    const size_t bm_words = (size_t)a.pitch * a.h;
    unsigned long long* key = reinterpret_cast<unsigned long long*>(ds_smem + ((bm_words * 4 + 15) & ~(size_t)15));
    unsigned short* order = reinterpret_cast<unsigned short*>(key + a.n_cells);
    uint8_t* span = reinterpret_cast<uint8_t*>(order + a.n_cells);
    const unsigned long long* K = a.cells + (size_t)frame * a.n_cells;

    const int max_new = a.max_new[frame];
    if (max_new <= 0) {                                                                 // ref: :71-72 early return
        if (tid == 0) { a.n_out[frame] = 0; a.exact[frame] = 0; }
        return;
    }
    if (tid == 0) { s_m = 0; s_tie = 0; }
    __syncthreads();
    // span table of every radius: span[r][|dy|] = half-width of row dy (OpenCV drawing.cpp, Circle with fill)
    if (tid <= kMaxRadius) {
        const int r = tid;
        uint8_t* sp = span + r * kSpanPitch;
        for (int k = 0; k <= r; ++k) sp[k] = 0;
        int err = 0, dx = r, dy = 0, plus = 1, minus = (r << 1) - 1;
        while (dx >= dy) {
            sp[dy] = (uint8_t)max((int)sp[dy], dx);
            sp[dx] = (uint8_t)max((int)sp[dx], dy);
            dy++;
            err += plus;
            plus += 2;
            const int mask = (err <= 0) - 1;
            err -= minus & mask;
            dx += mask;
            minus -= mask & 2;
        }
    }
    // bitmap from the mask image (bit set = not 255)
    const uint8_t* M = a.masks ? a.masks + (size_t)frame * a.w * a.h : nullptr;
    for (size_t i = tid; i < bm_words; i += kThreads) {
        unsigned v = 0;
        if (M) {
            const int y = (int)(i / a.pitch), x0 = 32 * (int)(i - (size_t)y * a.pitch);
            const uint8_t* row = M + (size_t)y * a.w;
            const int n = min(32, a.w - x0);
            for (int b = 0; b < n; ++b) v |= (__ldg(row + x0 + b) != 255 ? 1u : 0u) << b;
        }
        bm[i] = v;
    }
    // candidates above 20 as (score descending, cell) keys
    for (int i = tid; i < a.n_cells; i += kThreads) {
        const dsdtm_corner c = decode(K[i], a.seed);
        if (c.score > kMinScore) key[atomicAdd(&s_m, 1)] = ((unsigned long long)~__float_as_uint(c.score) << 32) | (unsigned)i;
    }
    __syncthreads();
    // prior circles: one warp per circle, one lane per row, concurrent circles overlap -> atomicOr
    if (a.circles) {
        const int nc = a.n_circles ? a.n_circles[frame] : 0;
        const dsdtm_circle* C = a.circles + (size_t)frame * a.circle_stride;
        const int warp = tid >> 5, lane = tid & 31;
        for (int q = warp; q < nc; q += kThreads / 32) {
            const dsdtm_circle ci = C[q];
            paint_rows(bm, a, span, __float2int_rn(ci.px[0]), __float2int_rn(ci.px[1]), ci.radius, lane, 32, true);   // cv::Point(Point2f)
        }
    }
    // rank by counting (keys are distinct: the cell index is in them); equal score bits = a tie
    const int m = s_m;
    for (int e = tid; e < m; e += kThreads) {
        const unsigned long long k = key[e];
        int rank = 0;
        bool tie = false;
        for (int q = 0; q < m; ++q) {
            const unsigned long long o = key[q];
            rank += o < k ? 1 : 0;
            tie |= (o >> 32) == (k >> 32) && o != k;
        }
        order[rank] = (unsigned short)(k & 0xFFFFu);
        if (tie) s_tie = 1;
    }
    __syncthreads();
    const bool literal = s_tie != 0;
    if (literal) {
        if (tid == 0) {
            Cand* cs = reinterpret_cast<Cand*>(key);
            for (int i = 0; i < a.n_cells; ++i) cs[i] = Cand{ decode(K[i], a.seed).score, i };
            std_sort(cs, (long)a.n_cells, [](const Cand& x, const Cand& y) { return y.score < x.score; });   // ref: :111
            int n = 0;
            for (int i = 0; i < a.n_cells; ++i)
                if (cs[i].score > kMinScore) order[n++] = (unsigned short)cs[i].cell;
        }
        __syncthreads();
    }
    if (tid >= 32) return;

    // the walk (ref: :125-150)
    const int lane = tid;
    dsdtm_corner* O = a.out + (size_t)frame * a.out_stride;
    int added = 0;
    for (int b0 = 0; b0 < m && added < max_new; b0 += 32) {
        const int e = b0 + lane;
        bool alive = e < m;
        dsdtm_corner c = dsdtm_corner{ 0, 0, 0, 0.f };
        if (alive) {
            c = decode(K[order[e]], a.seed);
            alive = !masked(bm, a.pitch, c.x, c.y);
        }
        while (added < max_new) {
            const unsigned bal = __ballot_sync(0xffffffffu, alive);
            if (!bal) break;
            const int w = __ffs(bal) - 1;
            const int wx = __shfl_sync(0xffffffffu, c.x, w), wy = __shfl_sync(0xffffffffu, c.y, w);
            if (lane == w) O[added] = c;                                                // ref: :145 Add_Feature
            ++added;
            paint_rows(bm, a, span, wx, wy, a.cell_size, lane, 32, false);             // ref: :146 circle(mask, p, CellSize, 0)
            __syncwarp();
            if (lane <= w) alive = false;
            else if (alive) alive = !masked(bm, a.pitch, c.x, c.y);
        }
        __syncwarp();
    }
    if (lane == 0) { a.n_out[frame] = added; a.exact[frame] = literal ? 1 : 0; }
}

size_t bitmap_bytes(const dsdtm_ctx* c) { return (size_t)(c->geo.w[0] + 31) / 32 * 4 * c->geo.h[0]; }

size_t smem_bytes(const dsdtm_ctx* c)   // bitmap | keys (8 bytes per cell) | order (2 bytes per cell) | span table
{
    return ((bitmap_bytes(c) + 15) & ~(size_t)15) + (size_t)c->n_cells * (8 + 2) + kSpanPitch * kSpanPitch;
}

}  // namespace

int detect_select_max_radius() { return kMaxRadius; }

// true when the context's geometry fits the kernel: the bitmap within kMaxBitmapBytes, cell indices within 16 bits, CellSize within
// the span table, and all of it within the opt-in shared memory of one CTA
bool detect_select_fits(const dsdtm_ctx* c, size_t max_smem)
{
    return bitmap_bytes(c) <= kMaxBitmapBytes && c->n_cells <= 65536 && c->prm.cell_size <= kMaxRadius && smem_bytes(c) <= max_smem;
}

cudaError_t launch_detect_select(dsdtm_ctx* c, int n, float seed, const uint8_t* masks_d, const dsdtm_circle* circles_d, int circle_stride,
                                 const int* n_circles_d, const int* max_new_d, dsdtm_corner* out_d, int out_stride, int* n_out_d,
                                 uint8_t* exact_d, cudaStream_t s)
{
    DetSelArgs a;
    a.cells = c->cells_d; a.n_cells = c->n_cells; a.seed = seed;
    a.w = c->geo.w[0]; a.h = c->geo.h[0]; a.pitch = (a.w + 31) / 32;
    a.cell_size = c->prm.cell_size;
    a.masks = masks_d; a.circles = circles_d; a.circle_stride = circle_stride; a.n_circles = n_circles_d;
    a.max_new = max_new_d; a.out = out_d; a.out_stride = out_stride; a.n_out = n_out_d; a.exact = exact_d;
    const size_t smem = smem_bytes(c);
    cudaError_t e = cudaFuncSetAttribute(detect_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    detect_select_kernel<<<n, kThreads, smem, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace dsdtm
