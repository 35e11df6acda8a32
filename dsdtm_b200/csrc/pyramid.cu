// pyramid.cu -- kernel (a): 8-bit Gaussian pyramid, cv::pyrDown semantics.
//
// Replaces Frame::ComputeImagePyramid (ref: src/Frame.cpp:74-81), i.e. cv::pyrDown on CV_8UC1 with default
// arguments: dst(y,x) = (sum_{i,j in [-2,2]} k_i k_j src(R(2y+i), R(2x+j)) + 128) >> 8, k = [1 4 6 4 1],
// R = BORDER_REFLECT_101, dst size ((w+1)/2, (h+1)/2). Integer arithmetic => bit-exact in any evaluation order.
//
// One launch per level over a batch of frames. Two kernels:
//   pyrdown_strip_kernel (levels with w % 8 == 0 and dw % 4 == 0, i.e. every level of 640x480 and the two big levels of
//   752x480): no shared memory. A thread owns 4 adjacent output columns and walks down a strip of RPT output rows with a
//   5-row sliding window held in registers. Per source row it issues one 8-byte and two 4-byte aligned loads (consecutive
//   lanes read consecutive 8-byte words: fully coalesced), does the horizontal [1 4 6 4 1] pass with two PRMT + four DP4A,
//   keeps the four 12-bit sums packed as 2 x u16 in two registers, and the vertical pass works on the packed pairs
//   (max 16 * 4080 = 65280 < 2^16: no carry between halves). One 32-bit store per 4 outputs.
//   pyrdown_tile_kernel (any size; odd / tiny levels): 64x16 output tile staged through shared memory with reflect-101.
// HBM-bound stage: algorithmic bytes per frame = sum_l (w_{l-1} h_{l-1} + w_l h_l) (SURVEY 8d: 510 000 B @640x480x5).
// Round-1 measurement (history in profiles/r1_pyramid_fast_align2d.md): the tile kernel alone ran at 600 GB/s = 9 % of HBM peak, issue-bound on
// byte-wide shared-memory traffic -- hence the register/DP4A strip kernel. (Fetching the 3 halo bytes from neighbouring lanes by
// shuffle instead of two extra L1-hit 4-byte loads was measured SLOWER: 0.384 vs 0.267 ms per 2072 frames.
// An 8-outputs-per-thread variant (one 16-byte load per row, 44 registers) and rows-per-thread 4/16/32 x unroll 2/4 were also
// measured: none beat 4 outputs x 8 rows x unroll 2 (0.498 ms per 4096 frames; see profiles/r1_pyramid_fast_align2d.md).)
#include "ctx.cuh"

namespace dsdtm {

namespace {

constexpr int TW = 64;               // output tile width
constexpr int TH = 16;               // output tile height
constexpr int SW = 2 * TW + 8;       // staged source columns: [2*x0-4, 2*x0+132)
constexpr int SH = 2 * TH + 3;       // staged source rows:    [2*y0-2, 2*y0+33)
constexpr int SWP = SW + 4;          // padded row pitch in bytes (multiple of 4)

__device__ __forceinline__ int reflect101(int i, int n)
{
    // valid for -n < i < 2n-1 (enough for a 5-tap kernel on n >= 3; n < 3 handled by the loop below)
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = (i < 0) ? -i : 2 * n - 2 - i;
    return i;
}

__global__ void __launch_bounds__(256) pyrdown_tile_kernel(uint8_t* __restrict__ frames, unsigned frame_stride, int first_slot,
                                                      const int* __restrict__ slots, unsigned src_off, unsigned dst_off,
                                                      int w, int h, int dw, int dh)
{
    __shared__ __align__(16) uint8_t s_src[SH][SWP];
    __shared__ uint16_t s_h[SH][TW];

    const int slot = slots ? slots[blockIdx.z] : first_slot + blockIdx.z;
    const uint8_t* __restrict__ src = frames + (size_t)slot * frame_stride + src_off;
    uint8_t* __restrict__ dst = frames + (size_t)slot * frame_stride + dst_off;

    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;
    const int sx0 = 2 * x0 - 4, sy0 = 2 * y0 - 2;
    const int tid = threadIdx.x;

    const bool fast = ((w & 3) == 0) && sx0 >= 0 && sx0 + SW <= w && sy0 >= 0 && sy0 + SH <= h;
    if (fast) {
        // coalesced 32-bit loads; (sy*w + sx0) is a multiple of 4 because w % 4 == 0 and sx0 % 4 == 0
        constexpr int WPR = SW / 4;
        for (int i = tid; i < SH * WPR; i += 256) {
            const int r = i / WPR, c = i - r * WPR;
            const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(src + (size_t)(sy0 + r) * w + sx0) + c);
            *reinterpret_cast<uint32_t*>(&s_src[r][4 * c]) = v;
        }
    } else {
        for (int i = tid; i < SH * SW; i += 256) {
            const int r = i / SW, c = i - r * SW;
            const int sy = reflect101(sy0 + r, h), sx = reflect101(sx0 + c, w);
            s_src[r][c] = __ldg(src + (size_t)sy * w + sx);
        }
    }
    __syncthreads();

    // horizontal pass: s_h[r][x] = sum_j k_j * s_src[r][2x + j + 4 - 2 .. ]   (window column of source col 2x0+2x-2 is 2x+2)
    for (int i = tid; i < SH * TW; i += 256) {
        const int r = i / TW, x = i - r * TW;
        const uint8_t* p = &s_src[r][2 * x + 2];
        s_h[r][x] = (uint16_t)(p[0] + 4 * p[1] + 6 * p[2] + 4 * p[3] + p[4]);
    }
    __syncthreads();

    // vertical pass: thread -> row ty, 4 consecutive outputs
    const int ty = tid >> 4, tx = (tid & 15) * 4;
    const int oy = y0 + ty, ox = x0 + tx;
    if (oy < dh && ox < dw) {
        uint32_t packed = 0;
        uint8_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int x = tx + k;
            const int s = s_h[2 * ty][x] + 4 * s_h[2 * ty + 1][x] + 6 * s_h[2 * ty + 2][x] + 4 * s_h[2 * ty + 3][x] + s_h[2 * ty + 4][x];
            o[k] = (uint8_t)((s + 128) >> 8);
            packed |= (uint32_t)o[k] << (8 * k);
        }
        uint8_t* q = dst + (size_t)oy * dw + ox;
        if (((dw & 3) == 0) && ox + 3 < dw) {
            *reinterpret_cast<uint32_t*>(q) = packed;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (ox + k < dw) q[k] = o[k];
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
#ifndef DSDTM_PYR_RPT
#define DSDTM_PYR_RPT 8
#endif
#ifndef DSDTM_PYR_UNROLL
#define DSDTM_PYR_UNROLL 2
#endif
constexpr int PYR_UNROLL = DSDTM_PYR_UNROLL;
constexpr int RPT = DSDTM_PYR_RPT;   // output rows per thread strip

__device__ __forceinline__ int reflect_row(int r, int h)
{
    r = (r < 0) ? -r : r;
    return (r >= h) ? 2 * h - 2 - r : r;
}

// horizontal pass of one source row for output columns x..x+3 (x % 4 == 0): returns the four sums packed as 2 x (2 x u16)
__device__ __forceinline__ uint2 hrow(const uint8_t* __restrict__ row, int x, int w)
{
    const int c0 = 2 * x;                                            // multiple of 8
    const uint2 mid = __ldg(reinterpret_cast<const uint2*>(row + c0));          // cols c0 .. c0+7
    const uint32_t w0 = mid.x, w1 = mid.y;
    // cols c0-2, c0-1 (reflect-101 at the left edge: -2 -> 2, -1 -> 1) in bytes 2,3 of wm1
    const uint32_t wm1 = (x > 0) ? __ldg(reinterpret_cast<const uint32_t*>(row + c0 - 4)) : __byte_perm(w0, 0, 0x1200);
    // col c0+8 (reflect-101 at the right edge: w -> w-2 = c0+6) in byte 0 of w2
    const uint32_t w2 = (c0 + 8 < w) ? __ldg(reinterpret_cast<const uint32_t*>(row + c0 + 8)) : (w1 >> 16);
    const uint32_t K = 0x04060401u;                                  // taps 1,4,6,4 on bytes 0..3; the fifth tap (1) is the addend
    const uint32_t h0 = __dp4a(__byte_perm(wm1, w0, 0x5432), K, (w0 >> 16) & 0xFFu);
    const uint32_t h1 = __dp4a(w0, K, w1 & 0xFFu);
    const uint32_t h2 = __dp4a(__byte_perm(w0, w1, 0x5432), K, (w1 >> 16) & 0xFFu);
    const uint32_t h3 = __dp4a(w1, K, w2 & 0xFFu);
    return make_uint2(h0 | (h1 << 16), h2 | (h3 << 16));
}

__global__ void __launch_bounds__(128) pyrdown_strip_kernel(uint8_t* __restrict__ frames, unsigned frame_stride, int first_slot,
                                                            const int* __restrict__ slots, unsigned src_off, unsigned dst_off,
                                                            int w, int h, int dw, int dh, int n_items)
{
    const int item = blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= n_items) return;
    const int xq = dw >> 2;                               // column groups per row
    const int strip = item / xq, x = (item - strip * xq) << 2;
    const int slot = slots ? slots[blockIdx.y] : first_slot + blockIdx.y;
    const uint8_t* __restrict__ src = frames + (size_t)slot * frame_stride + src_off;
    uint8_t* __restrict__ dst = frames + (size_t)slot * frame_stride + dst_off;
    const int y0 = strip * RPT;
    // window rows 2y-2 .. 2y+2
    uint2 r0 = hrow(src + (size_t)reflect_row(2 * y0 - 2, h) * w, x, w);
    uint2 r1 = hrow(src + (size_t)reflect_row(2 * y0 - 1, h) * w, x, w);
    uint2 r2 = hrow(src + (size_t)(2 * y0) * w, x, w);
#pragma unroll PYR_UNROLL
    for (int y = y0; y < min(y0 + RPT, dh); ++y) {
        const uint2 r3 = hrow(src + (size_t)reflect_row(2 * y + 1, h) * w, x, w);
        const uint2 r4 = hrow(src + (size_t)reflect_row(2 * y + 2, h) * w, x, w);
        // vertical [1 4 6 4 1] on packed u16 pairs, then (s + 128) >> 8 per half
        uint32_t a = r0.x + r4.x + 4u * (r1.x + r3.x) + 6u * r2.x + 0x00800080u;
        uint32_t b = r0.y + r4.y + 4u * (r1.y + r3.y) + 6u * r2.y + 0x00800080u;
        // bytes 1 and 3 of a / b are the four results
        *reinterpret_cast<uint32_t*>(dst + (size_t)y * dw + x) = __byte_perm(a, b, 0x7531);
        r0 = r2; r1 = r3; r2 = r4;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Bulk-staged kernel (levels whose source width is a multiple of 8 and whose output width is a multiple of 4): level images are dense, so the 2*TH+3 source rows
// of a tile of TH output rows are ONE contiguous byte range. One elected thread issues a single cp.async.bulk (TMA 1-D)
// for it and everybody waits on the mbarrier; memory latency is covered by the other resident CTAs (a tile is ~12-22 KB,
// 10-18 CTAs per SM), not by per-thread loads, and the arithmetic reads shared memory with immediate offsets: ~45
// instructions per 4 outputs instead of ~100 in the strip kernel, which was co-limited by issue slots (60 % busy at 52 % of
// DRAM throughput, profiles/r1_pyramid_fast_align2d.md).
#ifndef DSDTM_PYR_BULK_RPT
#define DSDTM_PYR_BULK_RPT 12       // output rows per thread (sweep: profiles/r1_pyramid_fast_align2d.md)
#endif
#ifndef DSDTM_PYR_BULK_THREADS
#define DSDTM_PYR_BULK_THREADS 160  // target CTA size; a tile is xq column groups x (threads / xq) sub-strips
#endif
constexpr int BRPT = DSDTM_PYR_BULK_RPT;
constexpr int BULK_PAD = 16;        // bytes in front of / behind the staged rows (edge threads read one word outside)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint2 hrow_s(const uint8_t* row, int c0, bool left, bool right)
{
    const uint2 mid = *reinterpret_cast<const uint2*>(row + c0);
    const uint32_t w0 = mid.x, w1 = mid.y;
    uint32_t wm1 = *reinterpret_cast<const uint32_t*>(row + c0 - 4);
    uint32_t w2 = *reinterpret_cast<const uint32_t*>(row + c0 + 8);
    if (left) wm1 = __byte_perm(w0, 0, 0x1200);          // reflect-101: cols -2, -1 -> 2, 1
    if (right) w2 = w1 >> 16;                            // col w -> w - 2
    const uint32_t K = 0x04060401u;
    const uint32_t h0 = __dp4a(__byte_perm(wm1, w0, 0x5432), K, __byte_perm(w0, 0, 0x4442));
    const uint32_t h1 = __dp4a(w0, K, __byte_perm(w1, 0, 0x4440));
    const uint32_t h2 = __dp4a(__byte_perm(w0, w1, 0x5432), K, __byte_perm(w1, 0, 0x4442));
    const uint32_t h3 = __dp4a(w1, K, __byte_perm(w2, 0, 0x4440));
    return make_uint2(__byte_perm(h0, h1, 0x5410), __byte_perm(h2, h3, 0x5410));
}

__global__ void __launch_bounds__(1024) pyrdown_bulk_kernel(uint8_t* __restrict__ frames, unsigned frame_stride, int first_slot,
                                                            const int* __restrict__ slots, unsigned src_off, unsigned dst_off,
                                                            int w, int h, int dw, int dh, int tile_rows)
{
    extern __shared__ __align__(128) uint8_t s_raw[];
    __shared__ __align__(8) unsigned long long s_bar;
    uint8_t* s_rows = s_raw + BULK_PAD;
    const int slot = slots ? slots[blockIdx.y] : first_slot + blockIdx.y;
    const uint8_t* __restrict__ src = frames + (size_t)slot * frame_stride + src_off;
    uint8_t* __restrict__ dst = frames + (size_t)slot * frame_stride + dst_off;
    const int ty0 = blockIdx.x * tile_rows, ty1 = min(ty0 + tile_rows, dh);
    const int lo = max(2 * ty0 - 2, 0), hi = min(2 * ty1, h - 1);            // source rows lo..hi: one contiguous range
    // the copy starts at an even row of a level whose width is a multiple of 8: 16-byte aligned; its size is rounded up to 16
    // bytes (an odd number of rows of a width that is 8 mod 16 ends on an 8-byte boundary) -- the extra 8 bytes are the next
    // row or, behind the last level, the zero padding of the slot
    const uint32_t bytes = ((uint32_t)(hi - lo + 1) * (uint32_t)w + 15u) & ~15u;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s_bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&s_bar)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(s_rows)), "l"(src + (size_t)lo * w), "r"(bytes), "r"(smem_u32(&s_bar)) : "memory");
    }
    // per-thread geometry while the copy is in flight
    const int xq = dw >> 2;
    const int strip = threadIdx.x / xq, g = threadIdx.x - strip * xq;
    const int c0 = 8 * g;
    const bool left = g == 0, right = g == xq - 1;
    const int y0 = ty0 + strip * BRPT, y1 = min(y0 + BRPT, ty1);
    {
        uint32_t done = 0;
        int spins = 0;
        while (!done) {
            asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                         : "=r"(done) : "r"(smem_u32(&s_bar)) : "memory");
            if (!done && ++spins > (1 << 22)) __trap();      // a lost copy must not hang the GPU
        }
    }
    if (y0 >= y1) return;
    const uint8_t* base = s_rows - (size_t)lo * w;       // base + r * w = staged source row r
    uint2 r0 = hrow_s(base + reflect_row(2 * y0 - 2, h) * w, c0, left, right);
    uint2 r1 = hrow_s(base + reflect_row(2 * y0 - 1, h) * w, c0, left, right);
    uint2 r2 = hrow_s(base + (2 * y0) * w, c0, left, right);
    uint8_t* out = dst + (size_t)y0 * dw + 4 * g;
#pragma unroll 2
    for (int y = y0; y < y1; ++y) {
        const uint2 r3 = hrow_s(base + reflect_row(2 * y + 1, h) * w, c0, left, right);
        const uint2 r4 = hrow_s(base + reflect_row(2 * y + 2, h) * w, c0, left, right);
        const uint32_t a = r0.x + r4.x + 4u * (r1.x + r3.x) + 6u * r2.x + 0x00800080u;
        const uint32_t b = r0.y + r4.y + 4u * (r1.y + r3.y) + 6u * r2.y + 0x00800080u;
        *reinterpret_cast<uint32_t*>(out) = __byte_perm(a, b, 0x7531);
        out += dw;
        r0 = r2; r1 = r3; r2 = r4;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Whole-level kernel for the SMALL ragged levels (752x480: 188x120 -> 94x60 -> 47x30, widths that are not multiples of 8): one CTA
// stages an entire source level in shared memory and keeps every level it produces there as the source of the next one, so the whole
// tail of the pyramid is one launch and one read of its first level. (The tile kernel's 64x16 tiles carry a 2.6x halo overhead at
// this size: 0.38 TB/s on these two levels = 45 % of the 752x480 pyramid's time.)
//   staging   one cp.async.bulk of the dense level (offsets are 16-byte aligned, the size is rounded up to 16 bytes into the slot's
//             zero padding) when its rows are 4-byte aligned (w % 4 == 0); byte loads into a 4-byte pitch otherwise
//   borders   only the LAST group of four output columns of a row touches columns >= w. Its 16 source bytes (columns c0 - 4 ..
//             c0 + 11, reflect-101 applied) are gathered once per row into an edge table; the thread that owns the last group reads the
//             table instead of the plane -- same instructions, different address, no divergence, no edge arithmetic in the loop
//   work      a thread owns one group of four output columns and a strip of output rows: the bulk kernel's register window
//             (4 LDS.32 + 4 DP4A per source row, vertical pass on packed u16 pairs). Round 1's warp-per-row separable form spent
//             33.9 k warp instructions per 752x480 frame on loop and index overhead for 8.5 k sums (94.6 us per 2048 frames, 6 % of
//             the pyramid's bytes in 35 % of its time: profiles/r1_euroc_sweep.md).
constexpr int SMALL_THREADS = 256;
constexpr int SMALL_SMEM_LIMIT = 96 * 1024;
constexpr int SMALL_PAD = 16;                // bytes in front of / behind every plane (group 0 reads one word in front, the last rows a few bytes behind)
__host__ __device__ constexpr int small_pitch(int w) { return (w + 3) & ~3; }

struct SmallChain {
    int n;                                   // levels produced by this launch
    int w[DSDTM_MAX_LEVELS], h[DSDTM_MAX_LEVELS];      // [0] = the staged source level, [i + 1] = the i-th produced level
    unsigned off[DSDTM_MAX_LEVELS];
    int a_bytes, b_bytes, e_bytes;           // shared-memory plan: pad | plane A | pad | plane B | pad | edge table | mbarrier
};

__device__ __forceinline__ uint2 hrow_e(const uint8_t* p, bool left)
{
    const uint32_t w0 = *reinterpret_cast<const uint32_t*>(p), w1 = *reinterpret_cast<const uint32_t*>(p + 4);
    const uint32_t w2 = *reinterpret_cast<const uint32_t*>(p + 8);
    uint32_t wm1 = *reinterpret_cast<const uint32_t*>(p - 4);
    if (left) wm1 = __byte_perm(w0, 0, 0x1200);          // reflect-101: cols -2, -1 -> 2, 1
    const uint32_t K = 0x04060401u;
    const uint32_t h0 = __dp4a(__byte_perm(wm1, w0, 0x5432), K, __byte_perm(w0, 0, 0x4442));
    const uint32_t h1 = __dp4a(w0, K, __byte_perm(w1, 0, 0x4440));
    const uint32_t h2 = __dp4a(__byte_perm(w0, w1, 0x5432), K, __byte_perm(w1, 0, 0x4442));
    const uint32_t h3 = __dp4a(w1, K, __byte_perm(w2, 0, 0x4440));
    return make_uint2(__byte_perm(h0, h1, 0x5410), __byte_perm(h2, h3, 0x5410));
}

// edge[r] = columns c0 - 4 .. c0 + 11 of row r, reflect-101 applied (columns the sums never use are clamped into the row)
__device__ __forceinline__ void small_fill_edge(uint32_t* edge, const uint8_t* plane, int pitch, int w, int h, int c0, int tid)
{
    for (int i = tid; i < 4 * h; i += SMALL_THREADS) {
        const uint8_t* row = plane + (i >> 2) * pitch;
        const int col0 = c0 - 4 + 4 * (i & 3);
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            int col = col0 + b;
            col = col < 0 ? -col : col;
            col = col >= w ? 2 * w - 2 - col : col;
            col = min(max(col, 0), w - 1);
            v |= (uint32_t)row[col] << (8 * b);
        }
        edge[i] = v;
    }
}

__global__ void __launch_bounds__(SMALL_THREADS) pyrdown_small_kernel(uint8_t* __restrict__ frames, unsigned frame_stride, int first_slot,
                                                                      const int* __restrict__ slots, const SmallChain ch)
{
    extern __shared__ __align__(128) uint8_t s_small[];
    uint8_t* s_a = s_small + SMALL_PAD;
    uint8_t* s_b = s_a + ch.a_bytes + SMALL_PAD;
    uint32_t* s_e = reinterpret_cast<uint32_t*>(s_b + ch.b_bytes + SMALL_PAD);
    unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(reinterpret_cast<uint8_t*>(s_e) + ch.e_bytes);
    const int slot = slots ? slots[blockIdx.x] : first_slot + blockIdx.x;
    uint8_t* __restrict__ frame = frames + (size_t)slot * frame_stride;
    const int tid = threadIdx.x;
    int pitch;                                                           // of the plane that holds the current source level
    {
        const int w = ch.w[0], h = ch.h[0];
        const uint8_t* __restrict__ src = frame + ch.off[0];
        if ((w & 3) == 0) {
            pitch = w;
            const uint32_t bytes = ((uint32_t)w * (uint32_t)h + 15u) & ~15u;
            if (tid == 0) {
                asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(s_bar)));
                asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            }
            __syncthreads();
            if (tid == 0) {
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(s_bar)), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"(smem_u32(s_a)), "l"(src), "r"(bytes), "r"(smem_u32(s_bar)) : "memory");
            }
            uint32_t done = 0;
            int spins = 0;
            while (!done) {
                asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n selp.u32 %0, 1, 0, p;\n}"
                             : "=r"(done) : "r"(smem_u32(s_bar)) : "memory");
                if (!done && ++spins > (1 << 22)) __trap();              // a lost copy must not hang the GPU
            }
        } else {
            pitch = small_pitch(w);
            const int lane = tid & 31, warp = tid >> 5;
            for (int r = warp; r < h; r += SMALL_THREADS / 32)
                for (int j = lane; j < w; j += 32) s_a[r * pitch + j] = __ldg(src + r * w + j);
            __syncthreads();
        }
    }
    uint8_t* cur = s_a;
    uint8_t* nxt = s_b;
    for (int l = 0; l < ch.n; ++l) {
        const int w = ch.w[l], h = ch.h[l], dw = ch.w[l + 1], dh = ch.h[l + 1];
        const int G = (dw + 3) >> 2;                                     // groups of four outputs per row
        small_fill_edge(s_e, cur, pitch, w, h, 8 * (G - 1), tid);
        __syncthreads();
        const int lanes = SMALL_THREADS / G;                             // strips that fit one pass of the CTA (0: more groups than threads)
        const int rpt = lanes > 0 ? (dh + lanes - 1) / lanes : dh;       // output rows per thread
        const int strips = (dh + rpt - 1) / rpt;
        uint8_t* __restrict__ dst = frame + ch.off[l + 1];
        const bool keep = l + 1 < ch.n;
        const int npitch = small_pitch(dw);
        for (int u = tid; u < G * strips; u += SMALL_THREADS) {
            const int strip = u / G, g = u - strip * G;
            const int y0 = strip * rpt, y1 = min(y0 + rpt, dh);
            const bool last = g == G - 1, left = g == 0 && !last;
            const uint8_t* base = last ? reinterpret_cast<const uint8_t*>(s_e) + 4 : cur + 8 * g;     // column c0 of row 0
            const int stride = last ? 16 : pitch;
            uint2 r0 = hrow_e(base + reflect_row(2 * y0 - 2, h) * stride, left);
            uint2 r1 = hrow_e(base + reflect_row(2 * y0 - 1, h) * stride, left);
            uint2 r2 = hrow_e(base + (2 * y0) * stride, left);
            const int x = 4 * g;
            for (int y = y0; y < y1; ++y) {
                const uint2 r3 = hrow_e(base + reflect_row(2 * y + 1, h) * stride, left);
                const uint2 r4 = hrow_e(base + reflect_row(2 * y + 2, h) * stride, left);
                const uint32_t a = r0.x + r4.x + 4u * (r1.x + r3.x) + 6u * r2.x + 0x00800080u;
                const uint32_t b = r0.y + r4.y + 4u * (r1.y + r3.y) + 6u * r2.y + 0x00800080u;
                const uint32_t out = __byte_perm(a, b, 0x7531);
                uint8_t* o = dst + y * dw + x;
                if ((dw & 3) == 0) {
                    *reinterpret_cast<uint32_t*>(o) = out;
                } else if ((dw & 1) == 0) {                              // rows start on 2-byte boundaries; x + 1 < dw whenever x < dw
                    *reinterpret_cast<uint16_t*>(o) = (uint16_t)out;
                    if (x + 2 < dw) *reinterpret_cast<uint16_t*>(o + 2) = (uint16_t)(out >> 16);
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (x + k < dw) o[k] = (uint8_t)(out >> (8 * k));
                }
                if (keep) *reinterpret_cast<uint32_t*>(nxt + y * npitch + x) = out;   // columns >= dw of the last group are never read as data
                r0 = r2; r1 = r3; r2 = r4;
            }
        }
        __syncthreads();
        uint8_t* t = cur; cur = nxt; nxt = t;      // the produced level is the next source
        pitch = npitch;
    }
}

// plans the chain of levels first .. that one CTA can produce from level first - 1; returns the number of levels (0: not eligible)
int plan_small_chain(const LevelGeom& g, int first, SmallChain& ch, size_t& smem)
{
    const int w0 = g.w[first - 1], h0 = g.h[first - 1];
    if (h0 < 3 || w0 < 3) return 0;
    ch.n = 0;
    ch.w[0] = w0; ch.h[0] = h0; ch.off[0] = g.off[first - 1];
    ch.a_bytes = (h0 * small_pitch(w0) + 15) & ~15;                     // the bulk copy's rounded-up size fits; every later plane that lands here is smaller
    ch.b_bytes = (g.h[first] * small_pitch(g.w[first]) + 15) & ~15;
    ch.e_bytes = 16 * h0;
    smem = (size_t)3 * SMALL_PAD + ch.a_bytes + ch.b_bytes + ch.e_bytes + 16;
    if (smem > (size_t)SMALL_SMEM_LIMIT) return 0;
    for (int l = first; l < g.levels; ++l) {
        if (g.h[l - 1] < 3 || g.w[l - 1] < 3) break;
        ch.w[ch.n + 1] = g.w[l]; ch.h[ch.n + 1] = g.h[l]; ch.off[ch.n + 1] = g.off[l];
        ch.n++;
    }
    return ch.n;
}

// the pyramid of n frames: one launch per level, except that one pyrdown_small_kernel launch builds a chain of small levels.
// With launch == false nothing is launched and only the count is returned (the launch tally of a replayed step, the profiler's).
int plan_levels(dsdtm_ctx* c, int first_slot, const int* slots_d, int n, cudaStream_t s, bool launch)
{
    const LevelGeom& g = c->geo;
    SmallChain chain;
    size_t chain_smem = 0;
    int launches = 0;
    for (int l = 1; l < g.levels; ++l, ++launches) {
        const int w = g.w[l - 1], h = g.h[l - 1], dw = g.w[l], dh = g.h[l];
        if ((w & 7) == 0 && (dw & 3) == 0 && h >= 3 && 2 * dw == w && (dw >> 2) <= 1024 && (size_t)(2 * BRPT + 3) * w + 2 * BULK_PAD + 16 <= 48 * 1024 && c->pyr_kernel == 0) {
            const int xq = dw >> 2;
            int strips = std::max(1, DSDTM_PYR_BULK_THREADS / xq);
            strips = std::min(strips, (dh + BRPT - 1) / BRPT);
            while (xq * strips > 1024) --strips;
            while (strips > 1 && (size_t)(2 * strips * BRPT + 3) * w + 2 * BULK_PAD + 16 > 48 * 1024) --strips;
            const int tile_rows = strips * BRPT;
            const size_t smem = (size_t)(2 * tile_rows + 3) * w + 2 * BULK_PAD + 16;   // + the round-up of the copy to 16 bytes
            dim3 grid((dh + tile_rows - 1) / tile_rows, n);
            if (launch) pyrdown_bulk_kernel<<<grid, xq * strips, smem, s>>>(c->frames_d, g.frame_stride, first_slot, slots_d, g.off[l - 1], g.off[l], w, h, dw, dh, tile_rows);
        } else if (c->pyr_kernel == 0 && plan_small_chain(g, l, chain, chain_smem) > 0) {
            if (launch) pyrdown_small_kernel<<<n, SMALL_THREADS, chain_smem, s>>>(c->frames_d, g.frame_stride, first_slot, slots_d, chain);
            l += chain.n - 1;                     // the chain produced levels l .. l + n - 1
        } else if ((w & 7) == 0 && (dw & 3) == 0 && h >= 3 && 2 * dw == w && c->pyr_kernel != 1) {
            const int n_items = (dw >> 2) * ((dh + RPT - 1) / RPT);
            dim3 grid((n_items + 127) / 128, n);
            if (launch) pyrdown_strip_kernel<<<grid, 128, 0, s>>>(c->frames_d, g.frame_stride, first_slot, slots_d, g.off[l - 1], g.off[l], w, h, dw, dh, n_items);
        } else {
            dim3 grid((dw + TW - 1) / TW, (dh + TH - 1) / TH, n);
            if (launch) pyrdown_tile_kernel<<<grid, 256, 0, s>>>(c->frames_d, g.frame_stride, first_slot, slots_d, g.off[l - 1], g.off[l], w, h, dw, dh);
        }
    }
    return launches;
}

cudaError_t launch_levels(dsdtm_ctx* c, int first_slot, const int* slots_d, int n, cudaStream_t s)
{
    c->launches += plan_levels(c, first_slot, slots_d, n, s, true);
    return cudaGetLastError();
}

}  // namespace

cudaError_t pyramid_init(dsdtm_ctx*) { return cudaFuncSetAttribute(pyrdown_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMALL_SMEM_LIMIT); }
cudaError_t launch_pyramid(dsdtm_ctx* c, int first_slot, int n, cudaStream_t s) { return launch_levels(c, first_slot, nullptr, n, s); }
cudaError_t launch_pyramid_slots(dsdtm_ctx* c, const int* slots_d, int n, cudaStream_t s) { return launch_levels(c, 0, slots_d, n, s); }
int pyramid_launches(dsdtm_ctx* c) { return plan_levels(c, 0, nullptr, 0, nullptr, false); }

}  // namespace dsdtm
