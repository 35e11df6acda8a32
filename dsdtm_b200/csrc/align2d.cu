// align2d.cu -- kernel (d): batched 2-D inverse-compositional patch alignment, an 8-lane group per 8x8 feature patch,
// and the affine patch warp that feeds it.
//
// align2d_kernel replaces Feature_Alignment::Align2DGaussNewton (ref: src/Feature_alignment.cpp:318-417), fp32 like the
// reference: H = sum J J^T over the 8x8 interior of the 10x10 bordered patch (exact in fp32: quarter-integers < 2^22),
// Hinv by the 3x3 cofactor formula (Eigen Matrix3f::inverse), then <= max_iters iterations of bilinear sampling,
// Jres accumulation and the (u, v, mean) update; converged iff du^2 + dv^2 < 0.03^2.
// Eight lanes per patch: lane (g, m) owns 8 pixels; the three Jres sums are reduced with an xor-shuffle tree (bitwise identical in
// every lane of the group => uniform control flow per patch). The reference sums the 64 terms sequentially in fp32, the tree
// differs: documented tolerance 1e-3 px on the refined position.
// Q4 (ref: :367-368 uses '>' where SVO uses '>='): with u_r == cols-4 or v_r == rows-4 the reference reads one byte past
// the row / image. We reproduce the linear addressing (next row's first pixel) and read bytes past the end of the level
// image as 0, identically in the oracle.
//
// warp_affine_kernel replaces Feature_Alignment::WarpAffine + GetPatchNoBoarder (ref: :206-275), one warp per candidate,
// fp32 non-contracted with the reference's operation order => bit-exact 10x10 uchar patches (incl. the integer-division
// quirk Q3: the sampling grid collapses to the reference pixel for search levels >= 1).
#include "ctx.cuh"
#include "cand_prep.cuh"

namespace dsdtm {

namespace {

struct A2dArgs {
    const uint8_t* frames; unsigned frame_stride; LevelGeom geo;
    const int* patch_slot;      // frame slot per patch
    const int* patch_level;     // < 0 = unused entry
    const uint8_t* patch10;     // n x 100
    const double* px_in;        // n x 2 start positions (level coordinates)
    double* px;                 // n x 2 refined positions
    uint8_t* conv;              // n
    int n, max_iters, patch0;
    const int* n_dev;           // optional: number of valid entries, known only on the device (entries past it are skipped)
    dsdtm_store_cand* store_out;   // optional: fold (px * 2^level, level, converged) into the map-store records (ref: :154-156)
};

constexpr int A2D_WARPS = 8;          // 8 warps = 32 patches per CTA
constexpr int A2D_PPW = 4;            // patches per warp: 8 lanes per patch

// v4: an 8-lane group per patch, four patches per warp. The per-patch scalar work (bilinear weights, Hinv * J, the update, the
// convergence test, loop control) is shared by four patches per warp instruction instead of two. Lane (g, m) = (l8 >> 2, l8 & 3)
// owns columns 2m, 2m + 1 and rows 4g .. 4g + 3 of the 8x8 interior; its taps are a 5 x 3 block (15 byte loads for 8 pixels), and
// both columns share one set of weights, so the per-pixel arithmetic runs as paired fp32 (FMUL2 / FADD2) on float2 (x = column 2m,
// y = column 2m + 1).
// Bit-equal to v3 (one half-warp per patch, lane = one column x four rows, xor butterfly 8, 4, 2, 1): every column is still summed
// sequentially over its four rows, and the tree below adds the same operands at every level -- xor 4 (row groups, v3's xor 8),
// xor 2 (columns c ^ 4, v3's xor 4), xor 1 (columns c ^ 2, v3's xor 2), then the two columns of a lane (v3's xor 1). IEEE addition
// is commutative, so both lanes of a pair hold the same value and control flow stays uniform per patch.
// No multiply-add is contracted: ptxas fuses FMUL2 -> FADD2 into FFMA2 even with the _rn intrinsics, so every product -> sum edge
// has exactly one paired side (tests/test_align2d_sass.py checks the SASS).
// Iterations on the bench batch are 2 or 3 for 99.8 % of the patches (profiles/r4_a2d_iter_hist.json): waiting for the slowest of
// four patches costs 7 % more lane-iterations than the slowest of two, far less than the amortised scalar work saves.
#ifndef DSDTM_A2D_MINB
#define DSDTM_A2D_MINB 3      // 80 registers, no spills (2 -> 101 registers; 4 -> 64 registers, 36 B spilled); per-cap times not measured
#endif
// reduce the three Jres sums of a patch (see above); on return every lane of the group holds the same three values
__device__ __forceinline__ float a2d_sum(float2 s, int g)
{
    s = __fadd2_rn(s, make_float2(__shfl_xor_sync(0xffffffffu, s.x, 4), __shfl_xor_sync(0xffffffffu, s.y, 4)));
    float v = g ? s.y : s.x;                              // column 2m + g: v3's xor 4 and xor 2 partners own the same parity
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 2));
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 4));   // even + odd columns (v3's xor 1)
}
__device__ __forceinline__ int a2d_sum_i(int v)
{
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }

__global__ void __launch_bounds__(A2D_WARPS * 32, DSDTM_A2D_MINB) align2d_kernel(const A2dArgs a)
{
    __shared__ __align__(16) uint8_t s_patch[A2D_WARPS * A2D_PPW][104];
    const int grp = threadIdx.x >> 3, l8 = threadIdx.x & 7, g = l8 >> 2, m = l8 & 3;
    const int n_eff = a.n_dev ? min(a.n, *a.n_dev) : a.n;
    const int last = a.patch0 + n_eff - 1;
    const int iraw = a.patch0 + blockIdx.x * (A2D_WARPS * A2D_PPW) + grp;
    if (iraw - (grp & (A2D_PPW - 1)) > last) return;      // whole warp out of range
    const bool exists = iraw <= last;
    const int i = exists ? iraw : last;                   // a missing group shadows the last patch and never writes
    const int L = a.patch_level[i];
    bool active = exists && L >= 0;
    if (exists && L < 0 && l8 == 0) { a.conv[i] = 0; a.px[2 * i] = a.px_in[2 * i]; a.px[2 * i + 1] = a.px_in[2 * i + 1]; }
    const int Lc = L < 0 ? 0 : L;

    // stage the 10x10 bordered patch (100 bytes = 25 words; patch10 rows are 4-byte aligned because 100 % 4 == 0)
    for (int q = l8; q < 25; q += 8)
        reinterpret_cast<uint32_t*>(s_patch[grp])[q] = __ldg(reinterpret_cast<const uint32_t*>(a.patch10 + (size_t)i * 100) + q);
    __syncwarp();

    // negated gradients and reference (exact): s - ref == s + (-ref) and j - res * d == j + res * (-d) bit for bit
    float2 ndx[4], ndy[4], nref[4];
    int i00 = 0, i01 = 0, i02 = 0, i11 = 0, i12 = 0;      // sums of the integer pixel differences (2*dx, 2*dy)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint8_t* it = s_patch[grp] + (4 * g + k + 1) * 10 + 1 + 2 * m;
        const int dx0 = (int)it[1] - (int)it[-1], dy0 = (int)it[10] - (int)it[-10];
        const int dx1 = (int)it[2] - (int)it[0], dy1 = (int)it[11] - (int)it[-9];
        ndx[k] = make_float2(-0.5f * (float)dx0, -0.5f * (float)dx1);        // ref: :336 (exact half-integers)
        ndy[k] = make_float2(-0.5f * (float)dy0, -0.5f * (float)dy1);        // ref: :337
        nref[k] = make_float2(-(float)it[0], -(float)it[1]);
        i00 += dx0 * dx0 + dx1 * dx1; i01 += dx0 * dy0 + dx1 * dy1; i02 += dx0 + dx1;
        i11 += dy0 * dy0 + dy1 * dy1; i12 += dy0 + dy1;
    }
    // H = sum J J^T with J = (dx, dy, 1): every entry is an integer / 4 (or / 2) below 2^22, exact in fp32 in any order
    const float h00 = 0.25f * (float)a2d_sum_i(i00), h01 = 0.25f * (float)a2d_sum_i(i01), h02 = 0.5f * (float)a2d_sum_i(i02);
    const float h11 = 0.25f * (float)a2d_sum_i(i11), h12 = 0.5f * (float)a2d_sum_i(i12);
    const float h22 = 64.0f;
    // Eigen 3x3 inverse: cofactor(i,j) = m(i1,j1) m(i2,j2) - m(i1,j2) m(i2,j1); det = sum_i cof(i,0) m(i,0)
    float Hinv[9];
    {
        const float m[9] = { h00, h01, h02, h01, h11, h12, h02, h12, h22 };
#define M(r, c) m[(r) * 3 + (c)]
#define COF(i, j) __fsub_rn(__fmul_rn(M(((i) + 1) % 3, ((j) + 1) % 3), M(((i) + 2) % 3, ((j) + 2) % 3)), \
                            __fmul_rn(M(((i) + 1) % 3, ((j) + 2) % 3), M(((i) + 2) % 3, ((j) + 1) % 3)))
        const float c00 = COF(0, 0), c10 = COF(1, 0), c20 = COF(2, 0);
        const float det = __fadd_rn(__fadd_rn(__fmul_rn(c00, M(0, 0)), __fmul_rn(c10, M(1, 0))), __fmul_rn(c20, M(2, 0)));
        // 1 / det rounded to fp64 and then to fp32 equals the fp32 quotient (double rounding is innocuous for a division when
        // 53 >= 2 * 24 + 2). __fdiv_rn's refinement would put FFMAs into the kernel's SASS; in inline PTX the compiler cannot
        // narrow the fp64 division back to it.
        double rdet;
        asm("div.rn.f64 %0, %1, %2;" : "=d"(rdet) : "d"(1.0), "d"((double)det));
        const float invdet = (float)rdet;
        Hinv[0] = __fmul_rn(c00, invdet); Hinv[1] = __fmul_rn(c10, invdet); Hinv[2] = __fmul_rn(c20, invdet);
        Hinv[3] = __fmul_rn(COF(0, 1), invdet); Hinv[4] = __fmul_rn(COF(1, 1), invdet); Hinv[5] = __fmul_rn(COF(2, 1), invdet);
        Hinv[6] = __fmul_rn(COF(0, 2), invdet); Hinv[7] = __fmul_rn(COF(1, 2), invdet); Hinv[8] = __fmul_rn(COF(2, 2), invdet);
#undef COF
#undef M
    }

    const int cols = a.geo.w[Lc], rows = a.geo.h[Lc];
    const uint8_t* __restrict__ img = a.frames + (size_t)a.patch_slot[i] * a.frame_stride + a.geo.off[Lc];
    const unsigned img_bytes = (unsigned)cols * (unsigned)rows;

    float u = (float)a.px_in[2 * i], v = (float)a.px_in[2 * i + 1];      // ref: :349-350
    float mean_diff = 0.f;
    const float min_update_squared = (float)(0.03 * 0.03);          // ref: :352
    bool converged = false;
    for (int it = 0; it < a.max_iters; ++it) {
        const float uf = floorf(u), vf = floorf(v);
        // ref: :367-369 (Q4 '>'); written on floats so that NaN / huge values break like the reference
        if (active && !(uf >= 4.f && vf >= 4.f && uf <= (float)(cols - 4) && vf <= (float)(rows - 4))) active = false;
        if (!__any_sync(0xffffffffu, active)) break;       // all four patches of the warp are done
        // a finished group keeps executing the (warp-wide) shuffles on clamped coordinates and discards the result
        const int u_r = active ? (int)uf : 4, v_r = active ? (int)vf : 4;
        const float sx = active ? u - uf : 0.f, sy = active ? v - vf : 0.f;
        const float wTL = (float)((1.0 - (double)sx) * (1.0 - (double)sy));   // ref: :373 (double arithmetic, narrowed)
        const float wTR = __fmul_rn(sx, 1.0f - sy);                          // ref: :374 (float arithmetic)
        const float wBL = (float)((1.0 - (double)sx) * (double)sy);          // ref: :375
        const float wBR = __fmul_rn(sx, sy);                                 // ref: :376
        const unsigned o0 = (unsigned)(v_r + 4 * g - 4) * (unsigned)cols + (unsigned)(u_r - 4 + 2 * m);
        // the whole 9x9 window lies inside the level image unless the Q4 edge case is hit (u_r == cols-4 or v_r == rows-4)
        const bool inside = (u_r + 4 < cols) && (v_r + 4 < rows);
        float2 tl[5], tr[5];                                // taps (2m, 2m+1) and (2m+1, 2m+2) of rows 4g .. 4g + 4
        if (inside) {
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const unsigned o = o0 + (unsigned)k * (unsigned)cols;
                const float p0 = (float)__ldg(img + o), p1 = (float)__ldg(img + o + 1), p2 = (float)__ldg(img + o + 2);
                tl[k] = make_float2(p0, p1); tr[k] = make_float2(p1, p2);
            }
        } else {                                            // ref: linear addressing, zeros past the end of the level image (Q4)
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                const unsigned o = o0 + (unsigned)k * (unsigned)cols;
                const float p0 = (float)(o < img_bytes ? __ldg(img + o) : 0);
                const float p1 = (float)(o + 1 < img_bytes ? __ldg(img + o + 1) : 0);
                const float p2 = (float)(o + 2 < img_bytes ? __ldg(img + o + 2) : 0);
                tl[k] = make_float2(p0, p1); tr[k] = make_float2(p1, p2);
            }
        }
        // paired products feed scalar sums (bilinear sample); scalar products feed paired sums (Jres): never both paired
        float2 j0 = f2(0.f), j1 = f2(0.f), j2 = f2(0.f);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 a0 = __fmul2_rn(f2(wTL), tl[k]), a1 = __fmul2_rn(f2(wTR), tr[k]);
            const float2 a2 = __fmul2_rn(f2(wBL), tl[k + 1]), a3 = __fmul2_rn(f2(wBR), tr[k + 1]);
            const float2 s = make_float2(__fadd_rn(__fadd_rn(__fadd_rn(a0.x, a1.x), a2.x), a3.x),
                                         __fadd_rn(__fadd_rn(__fadd_rn(a0.y, a1.y), a2.y), a3.y));          // ref: :386
            const float2 res = __fadd2_rn(__fadd2_rn(s, nref[k]), f2(mean_diff));                          // ref: :387
            j0 = __fadd2_rn(j0, make_float2(__fmul_rn(res.x, ndx[k].x), __fmul_rn(res.y, ndx[k].y)));
            j1 = __fadd2_rn(j1, make_float2(__fmul_rn(res.x, ndy[k].x), __fmul_rn(res.y, ndy[k].y)));
            j2 = make_float2(__fsub_rn(j2.x, res.x), __fsub_rn(j2.y, res.y));
        }
        const float J0 = a2d_sum(j0, g), J1 = a2d_sum(j1, g), J2 = a2d_sum(j2, g);
        // ref: :395 tUpdate = Hinv * Jres (row-wise, left to right)
        const float d0 = __fadd_rn(__fadd_rn(__fmul_rn(Hinv[0], J0), __fmul_rn(Hinv[1], J1)), __fmul_rn(Hinv[2], J2));
        const float d1 = __fadd_rn(__fadd_rn(__fmul_rn(Hinv[3], J0), __fmul_rn(Hinv[4], J1)), __fmul_rn(Hinv[5], J2));
        const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(Hinv[6], J0), __fmul_rn(Hinv[7], J1)), __fmul_rn(Hinv[8], J2));
        if (active) {
            u = __fadd_rn(u, d0); v = __fadd_rn(v, d1); mean_diff = __fadd_rn(mean_diff, d2);
            if (__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)) < min_update_squared) { converged = true; active = false; }   // ref: :400
        }
    }
    if (exists && L >= 0 && l8 == 0) {
        a.px[2 * i] = (double)u; a.px[2 * i + 1] = (double)v;     // ref: :414
        a.conv[i] = converged ? 1 : 0;
        if (a.store_out) {
            const double sc = (double)(1 << L);                   // ref: :154 tPt = tCurPx * (1 << tBestLevel) (exact)
            dsdtm_store_cand& o = a.store_out[i];
            o.r.px[0] = __dmul_rn((double)u, sc); o.r.px[1] = __dmul_rn((double)v, sc);
            o.r.level = L;
            if (converged) o.r.flags |= DSDTM_LM_CONVERGED;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
struct WaArgs {
    const uint8_t* frames; unsigned frame_stride; LevelGeom geo;
    const double* A;       // n x 4 row-major
    const float* ref_px;   // n x 2
    const int* meta;       // n x 3 : slot, ref_level, search_level
    uint8_t* out;          // n x 100
    int n;
    int i0;
    const int* n_dev;      // optional device-side count of valid entries
};

// A CTA owns WA_PPC consecutive candidates = WA_PPC * 100 consecutive output bytes. One lane per candidate derives the per-patch
// constants (the fp64 2x2 inverse with its division used to run on all 32 lanes of a warp per patch: a third of the kernel's
// instructions); then 320 threads walk the 1600 samples in 5 full rounds (a warp per patch left 100 samples on 32 lanes = 4 rounds at
// 78 % of the lanes). A thread keeps its patch column and steps two patch rows per round, so the loop has no division.
constexpr int WA_PPC = 16;
constexpr int WA_THREADS = 320;

__global__ void __launch_bounds__(WA_THREADS) warp_affine_kernel(const WaArgs a)
{
    __shared__ float s_f[WA_PPC][8];            // a00 a01 a10 a11 rx ry kf
    __shared__ int s_i[WA_PPC][4];              // w, h, valid
    __shared__ const uint8_t* s_img[WA_PPC];
    const int tid = threadIdx.x;
    const int first = a.i0 + blockIdx.x * WA_PPC;
    const int end = a.i0 + (a.n_dev ? min(a.n, *a.n_dev) : a.n);
    if (first >= end) return;
    if (tid < WA_PPC) {
        const int i = first + tid;
        int valid = 0;
        if (i < end) {
            const int slot = a.meta[3 * i], rl = a.meta[3 * i + 1], sl = a.meta[3 * i + 2];
            if (slot >= 0) {                                        // else: candidate skipped by candidate_prep_kernel
                valid = 1;
                const double A00 = a.A[4 * i], A01 = a.A[4 * i + 1], A10 = a.A[4 * i + 2], A11 = a.A[4 * i + 3];
                // Eigen 2x2 inverse in double, then cast<float>() (ref: :211)
                const double det = __dsub_rn(__dmul_rn(A00, A11), __dmul_rn(A10, A01));
                const double invdet = __ddiv_rn(1.0, det);
                s_f[tid][0] = (float)__dmul_rn(A11, invdet); s_f[tid][1] = (float)__dmul_rn(-A01, invdet);
                s_f[tid][2] = (float)__dmul_rn(-A10, invdet); s_f[tid][3] = (float)__dmul_rn(A00, invdet);
                s_f[tid][4] = __fdiv_rn(a.ref_px[2 * i], (float)(1 << rl));                    // ref: :215-216
                s_f[tid][5] = __fdiv_rn(a.ref_px[2 * i + 1], (float)(1 << rl));
                s_f[tid][6] = (float)(1 / (1 << sl));                                          // ref: :231 (Q3)
                s_i[tid][0] = a.geo.w[rl]; s_i[tid][1] = a.geo.h[rl];
                s_img[tid] = a.frames + (size_t)slot * a.frame_stride + a.geo.off[rl];
            }
        }
        s_i[tid][2] = valid;
    }
    __syncthreads();
    // sample s = tid + 320 k: patch s / 100, row (s % 100) / 10, column s % 10; 320 = 3 patches + 2 rows
    int p = tid / 100;
    const int j0 = tid - p * 100;
    int row = j0 / 10;
    const int col = j0 - row * 10;
    const float gx = (float)(col - 5);
    uint8_t* __restrict__ out = a.out + (size_t)first * 100 + tid;
#pragma unroll
    for (int k = 0; k < WA_PPC * 100 / WA_THREADS; ++k) {
        if (s_i[p][2]) {
            const float a00 = s_f[p][0], a01 = s_f[p][1], a10 = s_f[p][2], a11 = s_f[p][3], kf = s_f[p][6];
            const int w = s_i[p][0], h = s_i[p][1];
            const uint8_t* __restrict__ img = s_img[p];
            const float gy = (float)(row - 5);
            float wx = __fmul_rn(__fadd_rn(__fmul_rn(a00, gx), __fmul_rn(a01, gy)), kf);
            float wy = __fmul_rn(__fadd_rn(__fmul_rn(a10, gx), __fmul_rn(a11, gy)), kf);
            wx = __fadd_rn(wx, s_f[p][4]); wy = __fadd_rn(wy, s_f[p][5]);
            uint8_t o = 0;
            if (!(wx < 0 || wy < 0 || wx > (float)(w - 1) || wy > (float)(h - 1))) {       // ref: :249
                const int fx = __float2int_rd(wx), fy = __float2int_rd(wy);                // floor(): exact in either precision
                const float sx = __fsub_rn(wx, (float)fx), sy = __fsub_rn(wy, (float)fy);
                const float ox = __fsub_rn(1.0f, sx), oy = __fsub_rn(1.0f, sy);
                const float W00 = __fmul_rn(ox, oy), W01 = __fmul_rn(ox, sy), W10 = __fmul_rn(sx, oy);
                const float W11 = __fsub_rn(__fsub_rn(__fsub_rn(1.0f, W00), W01), W10);      // ref: :244
                const bool xin = fx + 1 < w, yin = fy + 1 < h;
                const uint8_t* q = img + fy * w + fx;
                const int p00 = __ldg(q);
                const int p01 = yin ? __ldg(q + w) : 0;
                const int p10 = xin ? __ldg(q + 1) : 0;
                const int p11 = (xin && yin) ? __ldg(q + w + 1) : 0;
                const float v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(W00, (float)p00), __fmul_rn(W01, (float)p01)), __fmul_rn(W10, (float)p10)),
                                          __fmul_rn(W11, (float)p11));                                                               // ref: :254-255
                o = (uint8_t)(int)v;   // truncating store
            }
            out[k * WA_THREADS] = o;
        }
        p += 3; row += 2;
        if (row >= 10) { row -= 10; ++p; }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// candidate_prep_kernel: SolveAffineMatrix + GetBestSearchLevel (ref: src/Feature_alignment.cpp:160-204), one thread per
// candidate, fp64 non-contracted in the reference's operation order (Eigen / Sophus semantics as in the oracle). Writes the
// inputs of warp_affine_kernel and align2d_kernel directly, so the three stages chain on the device.
__global__ void __launch_bounds__(128) candidate_prep_kernel(const CpArgs a)
{
    const int i = a.i0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.i0 + a.n) return;
    const dsdtm_candidate c = a.cand[i];
    candidate_prep_one(a, i, c, a.cur_slots ? a.cur_slots[i / a.ppp] : a.cur_slot);
}

}  // namespace

cudaError_t launch_candidate_prep(dsdtm_ctx* c, int n, int cur_slot, int max_search_level, cudaStream_t s, int i0, const int* cur_slots_d, int ppp)
{
    CpArgs a;
    a.cand = c->cand_d; a.n = n; a.cur_slot = cur_slot; a.max_search_level = max_search_level;
    a.i0 = i0; a.cur_slots = cur_slots_d; a.ppp = ppp > 0 ? ppp : 1;
    a.fx = c->cam.fx; a.fy = c->cam.fy; a.cx = c->cam.cx; a.cy = c->cam.cy;
    a.A = c->wa_A_d; a.ref_px = c->wa_px_d; a.meta = c->wa_meta_d; a.patch_level = c->patch_level_d; a.patch_slot = c->patch_slot_d;
    a.px_in = c->patch_px_in_d;
    candidate_prep_kernel<<<(n + 127) / 128, 128, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_align2d(dsdtm_ctx* c, int n_patches, int max_iters, cudaStream_t s, int patch0, const int* n_dev, dsdtm_store_cand* store_out)
{
    A2dArgs a;
    a.n_dev = n_dev; a.store_out = store_out;
    a.frames = c->frames_d; a.frame_stride = c->geo.frame_stride; a.geo = c->geo;
    a.patch_slot = c->patch_slot_d; a.patch_level = c->patch_level_d; a.patch10 = c->patches_d;
    a.px_in = c->patch_px_in_d; a.px = c->patch_px_d; a.conv = c->patch_conv_d; a.n = n_patches; a.max_iters = max_iters; a.patch0 = patch0;
    align2d_kernel<<<(n_patches + A2D_PPW * A2D_WARPS - 1) / (A2D_PPW * A2D_WARPS), A2D_WARPS * 32, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

cudaError_t launch_warp_affine(dsdtm_ctx* c, int n, uint8_t* out_d, cudaStream_t s, int i0, const int* n_dev)
{
    WaArgs a;
    a.i0 = i0; a.n_dev = n_dev;
    a.frames = c->frames_d; a.frame_stride = c->geo.frame_stride; a.geo = c->geo;
    a.A = c->wa_A_d; a.ref_px = c->wa_px_d; a.meta = c->wa_meta_d; a.out = out_d; a.n = n;
    warp_affine_kernel<<<(n + WA_PPC - 1) / WA_PPC, WA_THREADS, 0, s>>>(a);
    c->launches++;
    return cudaGetLastError();
}

}  // namespace dsdtm
