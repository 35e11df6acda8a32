// fast.cu -- kernel (b): FAST-10 detect + score + 3x3 non-max + Shi-Tomasi + per-cell argmax, all levels, one launch.
//
// Replaces the per-level body of Feature_detector::detect (ref: src/Feature_detection.cpp:76-109) and the FAST library
// it calls (ref: Thirdparty/fast/src/faster_corner_10_sse.cpp:15-202, fast_10_score.cpp:21-3147, nonmax_3x3.cpp:17-112):
//   detect : pixel is a corner at barrier b iff 10 contiguous ring pixels are all > p+b or all < p-b (strict)
//   score  : largest barrier at which it is still a corner = max_arc min_k |d_k| - 1   (closed form of the decision tree)
//   nonmax : keep iff every 8-neighbour corner has a strictly smaller score
//   cells  : Shi-Tomasi min-eigenvalue (fp32, non-contracted, same op order as the reference) and a packed 64-bit
//            atomicMax key per grid cell = (score bits << 32) | ~(level, y, x): highest score, earliest (level, raster) on ties,
//            which is exactly "replace iff strictly greater, visiting levels ascending in raster order" (ref: :104-107).
//
// Work decomposition (v2; v1 used one 512-thread CTA per tile with five __syncthreads phases and spent most of its time at
// those barriers, profiles/r1_pyramid_fast_align2d.md): one WARP per 32x16 tile of one level of one frame, four independent
// warps per CTA, no CTA barrier at all (tile table covers all levels, grid.y = frame). The 48x26 halo tile is
// staged in the warp's slice of shared memory with 8-byte row loads. Phase A rejects most pixels with the two opposite-pair
// tests (any 10-arc contains >= 1 of each opposite ring pair); survivors are compacted with ballot + popc into a small
// per-warp queue and phase B (ring masks, 10-arc bit test, closed-form score) runs on batches of 32 candidates, one per
// lane. Non-max walks the interior row by row (lane = column); every surviving corner is handled by the whole warp for
// Shi-Tomasi (64 pixels = 2 per lane; integer sums, exact in fp32 in any order) and one atomicMax.
#include "ctx.cuh"

namespace dsdtm {

namespace {

constexpr int FT_W = 30, FT_H = 16;        // interior tile: 30 wide so that interior + 1-px non-max ring = 32 columns = one lane each
constexpr int HALO = 5;                    // shi-tomasi needs +-5, fast score of the 1-px nonmax ring needs +-4
constexpr int SMP = 48;                    // staged row pitch = staged columns [xa, xa+48), xa = (x0-5) rounded down to 8
constexpr int SMH = FT_H + 2 * HALO;       // 26 staged rows (y0-5 .. y0+20)
constexpr int SC_H = FT_H + 2;             // score tile incl. 1-px ring: 32 (= FT_W + 2, one lane each) x 18
constexpr int SC_P = 32;                   // score row pitch
constexpr int WARPS = 4;
constexpr int QCAP = 64;
#ifndef DSDTM_FAST_UNROLL_A
#define DSDTM_FAST_UNROLL_A 1
#endif
constexpr int FAST_UNROLL_A = DSDTM_FAST_UNROLL_A;   // phase-A row-loop unroll (sweep in profiles/: 1, 2, 3 equal, 6 slower)

__constant__ int c_ring_dx[16] = { 0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1 };
__constant__ int c_ring_dy[16] = { 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3 };

__device__ __forceinline__ bool has_arc10(unsigned m)
{
    const unsigned d = m | (m << 16);
    unsigned r = d & (d >> 1);
    r &= r >> 2;
    r &= r >> 4;
    r &= d >> 8;
    r &= d >> 9;
    return (r & 0xFFFFu) != 0;
}

// max over the 16 cyclic 10-arcs of the minimum of v[] over the arc
__device__ __forceinline__ int max_arc_min10(const int (&v)[16])
{
    int m2[16], m4[16], best = -100000;
#pragma unroll
    for (int i = 0; i < 16; ++i) m2[i] = min(v[i], v[(i + 1) & 15]);
#pragma unroll
    for (int i = 0; i < 16; ++i) m4[i] = min(m2[i], m2[(i + 2) & 15]);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int m8 = min(m4[i], m4[(i + 4) & 15]);
        best = max(best, min(m8, m2[(i + 8) & 15]));
    }
    return best;
}

struct FastArgs {
    uint8_t* frames; unsigned frame_stride; int first_slot;
    const int* slots;                    // frame f reads slot slots[f], or first_slot + f when null
    const int* rows;                     // grid row y runs frame rows[y], or frame y when null
    const int* tiles; int n_tiles; LevelGeom geo;
    int barrier; float seed_score;
    const uint8_t* occupied;             // n * n_cells or null
    unsigned long long* cells;           // n * n_cells keys
    int n_cells, grid_cols, cell_size;
    unsigned cell_magic;                 // floor(2^32 / cell_size) + 1: exact x / cell_size for x < 65536 via __umulhi
    // score-map mode (parity helper): single level, dense outputs
    uint8_t* score_out; uint8_t* nonmax_out;
};

struct WarpSmem {
    uint8_t img[SMH][SMP];
    uint8_t score[SC_H][SC_P];
    unsigned short queue[QCAP];
};

// phase B for one candidate position i (index into the 18x34 score region)
__device__ __forceinline__ void score_candidate(WarpSmem& sm, int i, int b, int xoff)
{
    const int r = i >> 5, c = i & 31;
    const int sr = r + HALO - 1, sc = c + xoff - 1;
    const int p = sm.img[sr][sc];
    int d[16];
    unsigned bright = 0, dark = 0;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        d[k] = (int)sm.img[sr + c_ring_dy[k]][sc + c_ring_dx[k]] - p;
        bright |= (d[k] > b) ? (1u << k) : 0u;
        dark |= (d[k] < -b) ? (1u << k) : 0u;
    }
    const bool isb = has_arc10(bright);
    if (isb || has_arc10(dark)) {
        // score = max(S_bright, S_dark) - 1 with S = max over 10-arcs of min over the arc. Two 10-arcs of a 16-ring share at least
        // 4 pixels, so when a bright 10-arc exists every arc contains a brighter pixel and S_dark < 0 < S_bright (and vice versa):
        // only the polarity that made the pixel a corner has to be evaluated.
        if (!isb) {
#pragma unroll
            for (int k = 0; k < 16; ++k) d[k] = -d[k];
        }
        sm.score[r][c] = (uint8_t)(max_arc_min10(d) - 1);     // in [barrier, 254]
    }
}

__global__ void __launch_bounds__(32 * WARPS) fast_kernel(const FastArgs a)
{
    __shared__ __align__(16) WarpSmem s_all[WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x * WARPS + warp;
    if (tile >= a.n_tiles) return;
    WarpSmem& sm = s_all[warp];
    const int t = a.tiles[tile];
    const int L = t >> 24, tyi = (t >> 12) & 0xFFF, txi = t & 0xFFF;
    const int w = a.geo.w[L], h = a.geo.h[L];
    const int frame = a.rows ? a.rows[blockIdx.y] : (int)blockIdx.y;
    const int slot = a.slots ? a.slots[frame] : a.first_slot + frame;
    const uint8_t* __restrict__ img = a.frames + (size_t)slot * a.frame_stride + a.geo.off[L];
    const int x0 = txi * FT_W, y0 = tyi * FT_H;

    // ---- stage the halo tile: rows y0-5 .. y0+20, cols [xa, xa+48) with xa = (x0-5) & ~7 (zero outside the image)
    const int xa = (x0 - HALO) & ~7;           // arithmetic: -5 -> -8
    const int xoff = x0 - xa;                  // column of x0 inside the staged tile (5..12)
    if ((w & 7) == 0) {
        for (int i = lane; i < SMH * (SMP / 8); i += 32) {
            const int r = i / (SMP / 8), sgm = i - r * (SMP / 8);
            const int y = y0 - HALO + r, x = xa + 8 * sgm;
            uint2 v = make_uint2(0u, 0u);
            if (y >= 0 && y < h && x >= 0 && x < w) v = __ldg(reinterpret_cast<const uint2*>(img + (size_t)y * w + x));
            *reinterpret_cast<uint2*>(&sm.img[r][8 * sgm]) = v;
        }
    } else {
        for (int i = lane; i < SMH * SMP; i += 32) {
            const int r = i / SMP, c = i - r * SMP;
            const int y = y0 - HALO + r, x = xa + c;
            sm.img[r][c] = (x >= 0 && x < w && y >= 0 && y < h) ? __ldg(img + (size_t)y * w + x) : (uint8_t)0;
        }
    }
    for (int i = lane; i < SC_H * SC_P / 4; i += 32) reinterpret_cast<uint32_t*>(&sm.score[0][0])[i] = 0u;
    __syncwarp();

    // ---- phase A (quick reject; lane = column of the 32-wide score region, one row per iteration) + warp-level compaction
    //      + phase B on full batches of 32 candidates
    const int b = a.barrier;
    int qn = 0;
    {
        const int c = lane;
        const int x = x0 - 1 + c;
        const bool xok = x >= 3 && x < w - 3;                         // ref: fast_10.cpp:41 scan bounds
        const int sc = c + xoff - 1;
#pragma unroll FAST_UNROLL_A
        for (int r = 0; r < SC_H; ++r) {
            const int y = y0 - 1 + r;
            bool cand = false;
            if (xok && y >= 3 && y < h - 3) {                         // ref: fast_10.cpp:36
                const int sr = r + HALO - 1;
                const int p = sm.img[sr][sc];
                const int d0 = sm.img[sr + 3][sc] - p, d8 = sm.img[sr - 3][sc] - p;
                const int d4 = sm.img[sr][sc + 3] - p, d12 = sm.img[sr][sc - 3] - p;
                // bright: (d0 > b || d8 > b) && (d4 > b || d12 > b);  dark: the same with < -b
                cand = (min(max(d0, d8), max(d4, d12)) > b) || (max(min(d0, d8), min(d4, d12)) < -b);
            }
            const unsigned m = __ballot_sync(0xffffffffu, cand);
            if (cand) sm.queue[qn + __popc(m & ((1u << lane) - 1u))] = (unsigned short)(r * 32 + c);
            qn += __popc(m);
            __syncwarp();
            if (qn >= 32) {
                score_candidate(sm, sm.queue[lane], b, xoff);
                __syncwarp();
                const unsigned short carry = (lane < qn - 32) ? sm.queue[32 + lane] : (unsigned short)0;
                __syncwarp();
                if (lane < qn - 32) sm.queue[lane] = carry;
                qn -= 32;
                __syncwarp();
            }
        }
    }
    if (lane < qn) score_candidate(sm, sm.queue[lane], b, xoff);
    __syncwarp();

    // ---- non-max over the interior, row by row. Lane c owns score column c (0..31); a sliding 3-row window of its column
    //      lives in one register (3 bytes), the left / right columns arrive by shuffle. Interior columns are lanes 1..30.
    const int c = lane;
    const int x = x0 - 1 + c;
    unsigned col = (unsigned)sm.score[0][c] | ((unsigned)sm.score[1][c] << 8);      // rows r, r+1 of the window (bytes 0, 1)
    for (int r = 0; r < FT_H; ++r) {
        const int y = y0 + r;
        col |= (unsigned)sm.score[r + 2][c] << 16;                                  // byte 2 = row r+2
        const int s0 = col & 0xFF, s = (col >> 8) & 0xFF, s2 = (col >> 16) & 0xFF;
        const int own02 = max(s0, s2);                       // the two vertical neighbours
        const int col3 = max(own02, s);                      // column maximum, handed to the left / right lanes
        const int nb = max(max(__shfl_up_sync(0xffffffffu, col3, 1), __shfl_down_sync(0xffffffffu, col3, 1)), own02);
        const bool keep = (c >= 1) && (c <= FT_W) && s > 0 && x < w && y < h && nb < s;
        col >>= 8;
        if (a.score_out) {
            if (c >= 1 && c <= FT_W && x < w && y < h) {
                a.score_out[(size_t)y * w + x] = (uint8_t)s;
                a.nonmax_out[(size_t)y * w + x] = keep ? 1 : 0;
            }
            continue;
        }
        unsigned km = __ballot_sync(0xffffffffu, keep);
        while (km) {
            const int cc = __ffs(km) - 1;               // score column of the corner; image x = x0 - 1 + cc
            km &= km - 1;
            const int xx = x0 - 1 + cc;
            const int k = (int)__umulhi((unsigned)(y << L), a.cell_magic) * a.grid_cols + (int)__umulhi((unsigned)(xx << L), a.cell_magic);   // ref: Feature_detection.cpp:97-98
            if (a.occupied && a.occupied[(size_t)frame * a.n_cells + k]) continue;               // ref: :100
            float score = 0.f;
            // ref: :172 "patch too close to the boundary" -> 0
            if (!(xx - 4 < 1 || xx + 4 >= w - 1 || y - 4 < 1 || y + 4 >= h - 1)) {
                int sxx = 0, syy = 0, sxy = 0;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int pix = lane + 32 * e;                 // 8x8 box: rows y-4..y+3, cols x-4..x+3
                    const int sr = r + HALO - 4 + (pix >> 3), sc = cc - 1 + xoff - 4 + (pix & 7);
                    const int dx = (int)sm.img[sr][sc + 1] - (int)sm.img[sr][sc - 1];
                    const int dy = (int)sm.img[sr + 1][sc] - (int)sm.img[sr - 1][sc];
                    sxx += dx * dx; syy += dy * dy; sxy += dx * dy;
                }
                sxx = __reduce_add_sync(0xffffffffu, sxx);
                syy = __reduce_add_sync(0xffffffffu, syy);
                sxy = __reduce_add_sync(0xffffffffu, sxy);
                // |sums| <= 64*255^2 < 2^24: the reference's float accumulation is exact, so int -> float is the same value.
                // ref: :194-197, float arithmetic except the two double-typed constants (2.0*box_area = 128.0 and 0.5)
                const float dXX = (float)((double)(float)sxx / 128.0);
                const float dYY = (float)((double)(float)syy / 128.0);
                const float dXY = (float)((double)(float)sxy / 128.0);
                const float tr = __fadd_rn(dXX, dYY);
                const float disc = __fsub_rn(__fmul_rn(tr, tr), __fmul_rn(4.0f, __fsub_rn(__fmul_rn(dXX, dYY), __fmul_rn(dXY, dXY))));
                score = (float)(0.5 * (double)__fsub_rn(tr, __fsqrt_rn(disc)));
            }
            if (lane == 0 && score > a.seed_score) {
                const unsigned order = ((unsigned)L << 28) | ((unsigned)y << 14) | (unsigned)xx;
                const unsigned long long key = ((unsigned long long)__float_as_uint(score) << 32) | (unsigned long long)(~order);
                atomicMax(&a.cells[(size_t)frame * a.n_cells + k], key);
            }
        }
    }
}

FastArgs make_args(dsdtm_ctx* c, int first_slot)
{
    FastArgs a;
    a.frames = c->frames_d; a.frame_stride = c->geo.frame_stride; a.first_slot = first_slot;
    a.slots = nullptr; a.rows = nullptr;
    a.tiles = c->fast_tiles_d; a.n_tiles = c->n_fast_tiles; a.geo = c->geo;
    a.barrier = 20; a.seed_score = 0;
    a.occupied = nullptr; a.cells = c->cells_d; a.n_cells = c->n_cells; a.grid_cols = c->grid_cols; a.cell_size = c->prm.cell_size;
    a.cell_magic = (unsigned)(0x100000000ull / (unsigned)c->prm.cell_size) + 1u;
    a.score_out = nullptr; a.nonmax_out = nullptr;
    return a;
}

}  // namespace

// host: build the tile table (level << 24 | ty << 12 | tx) for all levels
int build_fast_tiles(const LevelGeom& g, int* out /* may be null: count only */, int* level_first /* levels+1 */)
{
    int n = 0;
    for (int l = 0; l < g.levels; ++l) {
        if (level_first) level_first[l] = n;
        const int tx = (g.w[l] + FT_W - 1) / FT_W, ty = (g.h[l] + FT_H - 1) / FT_H;
        for (int y = 0; y < ty; ++y)
            for (int x = 0; x < tx; ++x) {
                if (out) out[n] = (l << 24) | (y << 12) | x;
                ++n;
            }
    }
    if (level_first) level_first[g.levels] = n;
    return n;
}

cudaError_t launch_fast_cells(dsdtm_ctx* c, int first_slot, int n, int barrier, float seed_score, bool use_occupied, cudaStream_t s)
{
    cudaError_t e = cudaMemsetAsync(c->cells_d, 0, (size_t)n * c->n_cells * sizeof(unsigned long long), s);
    if (e != cudaSuccess) return e;
    FastArgs a = make_args(c, first_slot);
    a.barrier = barrier; a.seed_score = seed_score;
    a.occupied = use_occupied ? c->occupied_d : nullptr;
    dim3 grid((c->n_fast_tiles + WARPS - 1) / WARPS, n);
    fast_kernel<<<grid, 32 * WARPS, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

// the batched chain's key-frame detection: the n frames rows_d[0..n) (the wanted pairs), frame f on slot slots_d[f]; no memset of the cell
// keys (keyframe_seed_kernel zeroes the rows of the wanted frames inside the same step). Unwanted pairs get no CTA at all: an early return
// per CTA for every pair cost 0.48 ms per 4096 kinect pairs on a B200 at 1000 W (DESIGN §3i).
cudaError_t launch_fast_cells_slots(dsdtm_ctx* c, const int* slots_d, const int* rows_d, int n, float seed_score, cudaStream_t s)
{
    if (n == 0) return cudaSuccess;
    FastArgs a = make_args(c, 0);
    a.slots = slots_d; a.rows = rows_d;
    a.seed_score = seed_score;                   // barrier: the reference's literal 20 (ref: src/Feature_detection.cpp:81-82)
    a.occupied = c->occupied_d;
    dim3 grid((c->n_fast_tiles + WARPS - 1) / WARPS, n);
    fast_kernel<<<grid, 32 * WARPS, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_fast_score_map(dsdtm_ctx* c, int slot, int level, int barrier, cudaStream_t s)
{
    FastArgs a = make_args(c, slot);
    a.barrier = barrier;
    const LevelGeom& g = c->geo;
    a.score_out = c->scoremap_d;
    a.nonmax_out = c->scoremap_d + (size_t)g.w[0] * g.h[0];
    int first[DSDTM_MAX_LEVELS + 1];
    build_fast_tiles(g, nullptr, first);
    a.tiles = c->fast_tiles_d + first[level];
    a.n_tiles = first[level + 1] - first[level];
    dim3 grid((a.n_tiles + WARPS - 1) / WARPS, 1);
    fast_kernel<<<grid, 32 * WARPS, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace dsdtm
