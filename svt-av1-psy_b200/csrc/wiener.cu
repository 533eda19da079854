// wiener.cu -- K9 separable Wiener filter, K11 Wiener statistics (M = Y^T x, H = Y^T Y) (sm_100a).
//
// Reference behaviour restated:
//   svt_av1_wiener_convolve_add_src_c / svt_av1_highbd_wiener_convolve_add_src_c
//     (Source/Lib/Codec/convolve.c:100-147, 194-237 and the *_hip helpers :57-98, 149-192):
//     8-tap (7 + zero) horizontal pass with add-src, rounding round_0 and clamp to
//     WIENER_CLAMP_LIMIT, then vertical pass with add-src, rounding round_1 and pixel clip.
//   svt_av1_compute_stats_c / _highbd_c (Source/Lib/Codec/restoration_pick.c:659-745):
//     per pixel the wiener_win^2 window of (dgd - avg) is the vector y (column-major), x = src - avg;
//     M[k] += y[k] x, H[k][l] += y[k] y[l]; high bit depth divides by 4 / 16 at the end (truncating).
//
// B200 mapping of the statistics (the one dense contraction on the path):
//   8-bit pixels -> stats_mma_kernel: exact u8 x u8 -> s32 tcgen05 MMA on the raw pixels (see the comment above it);
//   10/12-bit    -> the lag-sum kernels of wiener_stats_lag.cuh (H[p][q] depends only on the lag between the two samples).
// The MMA kernel writes per-CTA int64 partials; stats_finalize_kernel adds them, folds the mean back in and mirrors
// the triangle.
#include <map>

#include "common.cuh"
#include "wiener_unit.cuh"
#include "../../include/svt_b200.h"
#include "wiener_stats_lag.cuh"

namespace b200 {


// ---------------------------------------------------------------------------------------------
// K9
// ---------------------------------------------------------------------------------------------
template <typename PIX>
__global__ void __launch_bounds__(256)
wiener_convolve_kernel(const PIX* __restrict__ src_base, PIX* __restrict__ dst_base, const SvtB200WienerUnit* __restrict__ units,
                       int n_units, int bd, int round0, int round1, int lbd_rows) {
    __shared__ __align__(16) uint16_t s_src[(64 + 8) * (64 + 8)];
    __shared__ __align__(16) uint16_t s_tmp[(64 + 8) * 64];
    for (int it = blockIdx.x; it < n_units; it += gridDim.x) {
        const SvtB200WienerUnit u = units[it];
        const int w = u.w, h = u.h;
        const PIX* src = src_base + u.src_off;
        PIX*       dst = dst_base + u.dst_off;
        const int sw = w + 8, sh = h + 7;  // rows -3..h+3, cols -3..w+4
#pragma unroll 4
        for (int i = threadIdx.x; i < sw * sh; i += blockDim.x) {
            const int r = i / sw, c = i - r * sw;
            // the 8th tap is read by the reference too (multiplied by its coefficient); the column
            // w+4 it touches on the last pixel is part of the caller's extended border
            s_src[r * 72 + c] = (uint16_t)src[(ptrdiff_t)(r - 3) * u.src_stride + (c - 3)];
        }
        __syncthreads();
        wiener_unit_compute<PIX>(s_src, s_tmp, dst, u.dst_stride, w, h, u.hfilter, u.vfilter, bd, round0, round1, lbd_rows);
    }
}

// ---------------------------------------------------------------------------------------------
// K11
// ---------------------------------------------------------------------------------------------
// Pixel total of every item's region (find_average, restoration_pick.c, divides it by w*h): kSumParts
// CTAs per item, one warp per row, totals combined with one 64-bit atomic per warp.
constexpr int kSumParts = 16;
template <typename PIX>
__global__ void __launch_bounds__(256)
stats_sum_kernel(const PIX* __restrict__ dgd_base, const SvtB200StatsItem* __restrict__ items, unsigned long long* __restrict__ tot_out) {
    const int it = blockIdx.x / kSumParts, part = blockIdx.x % kSumParts;
    const SvtB200StatsItem s = items[it];
    const int w = s.h_end - s.h_start, h = s.v_end - s.v_start;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned int acc = 0;  // <= (rows per warp) * (cols per lane) * 4095: far below 2^32 for any restoration unit
    unsigned long long wide = 0;
    for (int r = part * 8 + warp; r < h; r += kSumParts * 8) {
        const PIX* row = dgd_base + s.dgd_off + (ptrdiff_t)(s.v_start + r) * s.dgd_stride + s.h_start;
        for (int c = lane; c < w; c += 32) acc += row[c];
        if (acc > 0xf0000000u) { wide += acc; acc = 0; }
    }
    wide += acc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wide += __shfl_xor_sync(0xffffffffu, wide, o);
    if (lane == 0 && wide) atomicAdd(&tot_out[it], wide);
}

constexpr int kStatsMaxParts = 32;  // CTAs cooperating on one restoration unit

// ---------------------------------------------------------------------------------------------
// K11, 8-bit pixels: the contraction on the tensor cores (tcgen05.mma, kind::i8).
//
// The MMA runs on the RAW pixels (dgd - avg does not fit in 8 bits).  With G the Gram matrix of the raw window vectors,
// S_k the sum of window sample k over the region, Sx the source sum and n the pixel count, the reference's sums are
//   H_kl = G_kl - v (S_k + S_l) + n v^2,   M_k = G_kx - v S_k - v Sx + n v^2,   v = avg = S_centre / n
// (S_centre is the sum find_average divides by n), evaluated in int64 by stats_finalize_kernel.  u8 x u8 products
// (<= 255^2) accumulate in s32 tensor memory, exact for kTcFoldPixels pixels; past that the CTA folds TMEM into its
// int64 partial.  Bit-exact with the reference for any input; tests/test_wiener.py holds the extremes.
//
// Operand (K = pixels, 32 per MMA; a tile = up to kTcTW pixels of stats_tile_rows(WIN) rows): for every image row r of
// the tile (tile rows -WIN/2 .. last + WIN/2) the CTA writes one 8-row GROUP: row dx < WIN is dgd row r shifted by
// dx - WIN/2, row 7 is src row r; columns past the region's width are zero in every row.  Layout: K-major, no swizzle,
// 16-byte core-matrix rows, LBO = 128 B along K, SBO = kTcGrpBytes between groups.  One descriptor starting at the group
// of row y - WIN/2 is both A and B of an M = N = 128 MMA (16 groups), so with a = 8 dy + dx
//   D[a + 8t][b + 8t] = sum over the MMA's 32 pixels of output row y + t of  (window sample a) * (window sample b):
// the window products of T = stats_block_rows(WIN) consecutive output rows at once, on the 8-row diagonals of D
// (column b = 8 (WIN/2) + 7 is the source sample: G_kx).  A tile issues one MMA per block of T rows and 32 pixels; the
// readback sums G(a, b) = sum_t D[a + 8t][b + 8t].  D row i is TMEM lane i (PTX ISA data-path layout for M = 128,
// cta_group::1); the entries off those diagonals are don't-care.  Blocks run into a D at TMEM column 0; the short last
// block of a region's bottom tiles runs into a second D at column 128 whose diagonals are summed over its own row count.
// S_k and Sx come from per-(group, row) byte sums (DP4A) taken while the groups are written.
//
// One elected thread issues the MMAs of a tile and commits them to the buffer's mbarrier; the other threads build
// the next tile into the second buffer meanwhile.
constexpr int kTcThreads = 128;
constexpr int kTcTW = 128;                                 // pixels per tile row (4 K-steps)
// output rows whose window products one M = N = 128 MMA holds (a + 8t < 128 for every needed a = 8 dy + dx: 10, 12, 14),
// and the rows of a tile: a whole number of blocks, at most 36
__host__ __device__ constexpr int stats_block_rows(int win) { return (127 - 9 * (win - 1)) / 8 + 1; }
__host__ __device__ constexpr int stats_tile_rows(int win) { return stats_block_rows(win) * (36 / stats_block_rows(win)); }
constexpr int kTcGrpBytes = 8 * 128 + 16;                  // +16: the 8 groups a quarter warp writes land on distinct banks
constexpr int kTcGroups = 40;                              // every WIN: >= rows + WIN - 1 written, >= rows - T + 16 read
constexpr int kTcBufBytes = kTcGroups * kTcGrpBytes;
constexpr int kTcRowSums = kTcGroups * 8;                  // byte sum of every (group, row) of a tile
constexpr int kTcDumpPitch = 129;                          // words per D row when D is read back through shared memory
constexpr int kTcSmem = 2 * kTcBufBytes + 2 * kTcRowSums * 4 + 32;
constexpr int kTcFoldPixels = 33025;                       // 2^31 / 255^2: the s32 accumulators stay exact
constexpr int kTcTmemCols = 256;                           // two 128-column D
constexpr bool stats_tc_fits(int win) {
    return stats_tile_rows(win) + win - 1 <= kTcGroups && stats_tile_rows(win) - stats_block_rows(win) + 16 <= kTcGroups;
}
static_assert(stats_tc_fits(7) && stats_tc_fits(5) && stats_tc_fits(3), "operand buffer");
static_assert(128 * kTcDumpPitch * 4 <= 2 * kTcBufBytes, "D is read back through the operand buffers");
static_assert(kTcBufBytes % 16 == 0 && kTcSmem < 227 * 1024 / 2, "two CTAs per SM (2 x 256 TMEM columns)");

// per-CTA partial (int64 words): the upper triangle of G by reference index (row p holds columns q >= p), G_kx, S_k, Sx
// and n -- everything exact, combined and expanded by stats_finalize_kernel
constexpr int kPartG = 0, kPartGx = 1225, kPartS = kPartGx + 49, kPartSx = kPartS + 49, kPartN = kPartSx + 1;
constexpr int kStatsPartWords = kPartN + 1;
constexpr size_t kStatsItemWords = (size_t)kStatsMaxParts * kStatsPartWords;  // scratch words per item (either path)
static_assert(kStatsItemWords >= (size_t)kLagItemWords, "the lag path shares the scratch");

__host__ __device__ __forceinline__ int stats_tri_index(int w2, int p, int q) { return p * w2 - p * (p - 1) / 2 + q - p; }
// CTAs of an item that actually get pixel tiles (and so write a partial)
__device__ __forceinline__ int stats_mma_parts(const SvtB200StatsItem& s, int ctas_per_item) {
    const int th = stats_tile_rows(s.wiener_win);
    const int tiles = ((s.h_end - s.h_start + kTcTW - 1) / kTcTW) * ((s.v_end - s.v_start + th - 1) / th);
    return tiles < ctas_per_item ? tiles : ctas_per_item;
}

__device__ __forceinline__ uint32_t tc_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_bar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(tc_smem(bar)), "r"(parity) : "memory");
    } while (!ok);
}
// shared-memory matrix descriptor: start >> 4, LBO = 128 B, SBO = kTcGrpBytes, descriptor version 1 (bit 46), no swizzle
__device__ __forceinline__ uint64_t tc_desc(uint32_t addr) {
    return (uint64_t)((addr >> 4) & 0x3fffu) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(kTcGrpBytes >> 4) << 32) | (1ull << 46);
}
// instruction descriptor of kind::i8: D s32 (bits 4-5 = 2), A and B unsigned (bits 7-9, 10-12 = 0), both K-major,
// N >> 3 at bit 17, M >> 4 at bit 24
template <int N>
__host__ __device__ constexpr uint32_t tc_idesc() { return (2u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24); }
__device__ __forceinline__ void tc_mma_i8(uint32_t tmem, uint64_t desc, uint32_t idesc, uint32_t accum) {
    asm volatile("{ .reg .pred p; setp.ne.b32 p, %3, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %1, %2, p; }"
                 ::"r"(tmem), "l"(desc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Writes the groups of one tile into `op` and adds their per-(group, row) byte sums to `rs` (zeroed).  Only the
// 16-byte chunks of the K-steps that will be issued are written; a chunk past the region's width is written as zeros.
template <int WIN>
__device__ __forceinline__ void tc_build(uint8_t* __restrict__ op, int* __restrict__ rs, const uint8_t* __restrict__ dgd,
                                         const uint8_t* __restrict__ src, int dgd_stride, int src_stride, int r0, int c0, int nrows,
                                         int ncols) {
    constexpr int HALF = WIN / 2;
    constexpr uint32_t ONES = 0x01010101u;
    const int ng = nrows + WIN - 1, nkc = ((ncols + 31) >> 5) * 2;
    for (int c = threadIdx.x; c < ng * nkc; c += kTcThreads) {
        const int kc = c / ng, g = c - kc * ng;            // a quarter warp: 8 consecutive groups, one chunk
        const int kv = min(max(ncols - 16 * kc, 0), 16);   // columns of the region in this chunk
        uint32_t mask[4];
#pragma unroll
        for (int m = 0; m < 4; m++) {
            const int vb = min(max(kv - 4 * m, 0), 4);
            mask[m] = vb == 4 ? 0xffffffffu : (1u << (8 * vb)) - 1u;
        }
        uint8_t* dst = op + g * kTcGrpBytes + kc * 128;
        int*     rsg = rs + g * 8;
        const int r = r0 - HALF + g;
        // dgd bytes [a, a + kv + WIN - 1) with a = column c0 - HALF + 16 kc: the aligned words holding one of them
        const uint8_t*  p   = dgd + (ptrdiff_t)r * dgd_stride + (c0 - HALF + 16 * kc);
        const uint32_t  off = (uint32_t)(uintptr_t)p & 3u;
        const uint32_t* wp  = reinterpret_cast<const uint32_t*>(p - off);
        const int       nw  = kv ? (int)(off + kv + WIN + 2) >> 2 : 0;
        uint32_t w[7], u[6];
#pragma unroll
        for (int i = 0; i < 7; i++) w[i] = i < nw ? __ldg(wp + i) : 0u;
#pragma unroll
        for (int i = 0; i < 6; i++) u[i] = __funnelshift_r(w[i], w[i + 1], off * 8);  // bytes a + 4i ..
#pragma unroll
        for (int dx = 0; dx < WIN; dx++) {
            uint32_t o[4];
#pragma unroll
            for (int m = 0; m < 4; m++) o[m] = __funnelshift_r(u[(dx >> 2) + m], u[(dx >> 2) + m + 1], (dx & 3) * 8) & mask[m];
            *reinterpret_cast<uint4*>(dst + dx * 16) = make_uint4(o[0], o[1], o[2], o[3]);
            const uint32_t sum = __dp4a(o[0], ONES, __dp4a(o[1], ONES, __dp4a(o[2], ONES, __dp4a(o[3], ONES, 0u))));
            if (sum) atomicAdd(&rsg[dx], (int)sum);
        }
        if (g >= HALF && g < HALF + nrows) {  // row 7: the source row (only the tile's own rows are ever used)
            const uint8_t*  q    = src + (ptrdiff_t)r * src_stride + c0 + 16 * kc;
            const uint32_t  off2 = (uint32_t)(uintptr_t)q & 3u;
            const uint32_t* wq   = reinterpret_cast<const uint32_t*>(q - off2);
            const int       nw2  = kv ? (int)(off2 + kv + 3) >> 2 : 0;
            uint32_t x[5], o[4];
#pragma unroll
            for (int i = 0; i < 5; i++) x[i] = i < nw2 ? __ldg(wq + i) : 0u;
#pragma unroll
            for (int m = 0; m < 4; m++) o[m] = __funnelshift_r(x[m], x[m + 1], off2 * 8) & mask[m];
            *reinterpret_cast<uint4*>(dst + 7 * 16) = make_uint4(o[0], o[1], o[2], o[3]);
            const uint32_t sum = __dp4a(o[0], ONES, __dp4a(o[1], ONES, __dp4a(o[2], ONES, __dp4a(o[3], ONES, 0u))));
            if (sum) atomicAdd(&rsg[7], (int)sum);
        }
    }
}

template <int WIN>
__device__ __forceinline__ void stats_tc_body(const uint8_t* __restrict__ dgd, const uint8_t* __restrict__ src, const SvtB200StatsItem& s,
                                              const int part, const int parts, long long* __restrict__ P, uint8_t* smem) {
    constexpr int HALF = WIN / 2, W2 = WIN * WIN, T = stats_block_rows(WIN), TH = stats_tile_rows(WIN);
    constexpr uint32_t IDESC = tc_idesc<128>();
    // the S loop below reads row sums up to group TH - 1 + WIN - 1, row 7 (window rows dy < WIN; Sx: dy = WIN/2, row 7)
    static_assert((TH - 1 + WIN - 1) * 8 + 7 < kTcRowSums, "row sums of a tile");
    int*      rsum  = reinterpret_cast<int*>(smem + 2 * kTcBufBytes);  // [2][kTcRowSums]
    uint64_t* bar   = reinterpret_cast<uint64_t*>(rsum + 2 * kTcRowSums);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(bar + 2);
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&bar[0])) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(tc_smem(&bar[1])) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 2 * kTcRowSums; i += kTcThreads) rsum[i] = 0;
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(tslot)), "r"(kTcTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tslot;

    const int W = s.h_end - s.h_start, H = s.v_end - s.v_start;
    const int ntx = (W + kTcTW - 1) / kTcTW, nty = (H + TH - 1) / TH, ntiles = ntx * nty;
    const int rlast = (H - (nty - 1) * TH) % T;  // rows of the short last block of the bottom tiles (0: none)
    // D (128 x 128 s32 at TMEM column col) -> shared memory (over the operand buffers), then the partial's G and G_kx
    // entries (+)= sum over t < nt of D[a + 8t][b + 8t].  Every thread; the tensor core has finished.
    auto drain_one = [&](uint32_t col, int nt, bool add) {
        int* d = reinterpret_cast<int*>(smem);
#pragma unroll 1
        for (int c = 0; c < 128; c += 16) {
            uint32_t v[16];
            tc_ld16(tmem + ((uint32_t)(warp * 32) << 16) + col + (uint32_t)c, v);
#pragma unroll
            for (int j = 0; j < 16; j++) d[tid * kTcDumpPitch + c + j] = (int)v[j];
        }
        __syncthreads();
        for (int e = tid; e < W2 * W2 + W2; e += kTcThreads) {
            int p, b;
            long long* dst;
            if (e < W2 * W2) {
                p = e / W2;
                const int q = e - p * W2;
                if (q < p) continue;
                b   = 8 * (q % WIN) + q / WIN;  // reference index q = dx * WIN + dy -> D index 8 dy + dx
                dst = P + kPartG + stats_tri_index(W2, p, q);
            } else {
                p   = e - W2 * W2;
                b   = 8 * HALF + 7;
                dst = P + kPartGx + p;
            }
            const int  a = 8 * (p % WIN) + p / WIN;
            long long  g = 0;
            const int* dd = d + a * kTcDumpPitch + b;
            for (int t = 0; t < nt; t++) g += dd[t * (8 * kTcDumpPitch + 8)];
            *dst = (add ? *dst : 0) + g;
        }
        __syncthreads();
    };
    bool full_used = false, part_used = false;  // D at column 0 / 128 holds products since the start or the last fold
    auto drain = [&](bool add) {
        if (full_used) {
            drain_one(0, T, add);
            add = true;
        }
        if (part_used) drain_one(128, rlast, add);
    };

    // thread i < 64 with (dy, dx) = (i / 8, i % 8) both < WIN sums S of that window sample, reference index dx * WIN + dy;
    // thread 8 HALF + 7, the source row of the centre group, sums Sx.  No other thread reads the row sums.
    const int  dy = tid >> 3, dx = tid & 7, pidx = dx * WIN + dy;
    const bool wlane = dy < WIN && dx < WIN, slane = wlane || tid == 8 * HALF + 7;
    long long  ssum = 0, npix = 0;
    int        pending = 0;               // pixels in the s32 accumulators
    bool       spilled = false;           // the partial already holds folded totals
    uint32_t   inflight = 0, phase = 0;   // per buffer (bit b): MMAs committed and not yet waited for; barrier parity
    auto wait_buf = [&](int b) {
        if (inflight >> b & 1u) {
            tc_bar_wait(&bar[b], phase >> b & 1u);
            phase ^= 1u << b;
            inflight &= ~(1u << b);
        }
    };
    for (int tl = part, j = 0; tl < ntiles; tl += parts, j++) {
        const int b  = j & 1;
        const int ty = tl / ntx, tx = tl - ty * ntx;
        const int r0 = s.v_start + ty * TH, c0 = s.h_start + tx * kTcTW;
        const int nrows = min(TH, s.v_end - r0), ncols = min(kTcTW, s.h_end - c0);
        __syncthreads();  // the zeroing of rsum[b] (previous tile) is done
        if (pending + nrows * ncols > kTcFoldPixels) {  // CTA-uniform
            wait_buf(b ^ 1);                            // the previous tile's MMAs and, with them, every earlier one
            tc_fence_after();
            drain(spilled);
            tc_fence_before();
            spilled   = true;
            full_used = part_used = false;
            pending   = 0;
        }
        wait_buf(b);  // the tensor core no longer reads this buffer
        uint8_t* op = smem + b * kTcBufBytes;
        int*     rs = rsum + b * kTcRowSums;
        tc_build<WIN>(op, rs, dgd, src, s.dgd_stride, s.src_stride, r0, c0, nrows, ncols);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads
        __syncthreads();
        if (tid == 0) {
            tc_fence_after();
            const uint64_t d0 = tc_desc(tc_smem(op));
            const int      nk = (ncols + 31) >> 5;
            for (int y = 0; y < nrows; y += T) {
                const bool full = y + T <= nrows;
                bool&      used = full ? full_used : part_used;
                for (int k = 0; k < nk; k++) {
                    tc_mma_i8(tmem + (full ? 0u : 128u), d0 + (uint64_t)((y * kTcGrpBytes + k * 256) >> 4), IDESC, used ? 1u : 0u);
                    used = true;
                }
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(tc_smem(&bar[b])) : "memory");
        } else {  // the same bookkeeping in every thread (CTA-uniform: drain() depends on it)
            if (nrows >= T) full_used = true;
            if (nrows % T) part_used = true;
        }
        inflight |= 1u << b;
        if (slane) {  // S of this tile: the row sums of groups dy .. dy + nrows - 1, row dx
            int t = 0;
            for (int y = 0; y < nrows; y++) t += rs[(y + dy) * 8 + dx];
            ssum += t;
        }
        __syncthreads();
        for (int i = tid; i < kTcRowSums; i += kTcThreads) rs[i] = 0;
        pending += nrows * ncols;
        npix += nrows * ncols;
    }
    wait_buf(0);
    wait_buf(1);
    tc_fence_after();
    drain(spilled);
    if (wlane) P[kPartS + pidx] = ssum;
    if (tid == 8 * HALF + 7) P[kPartSx] = ssum;
    if (tid == 0) P[kPartN] = npix;
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTcTmemCols) : "memory");
    }
}

__global__ void __launch_bounds__(kTcThreads)
stats_mma_kernel(const uint8_t* __restrict__ dgd_base, const uint8_t* __restrict__ src_base, const SvtB200StatsItem* __restrict__ items,
                 int ctas_per_item, long long* __restrict__ partial) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int it = blockIdx.x / ctas_per_item, part = blockIdx.x % ctas_per_item;
    const SvtB200StatsItem s = items[it];
    if (part >= stats_mma_parts(s, ctas_per_item)) return;  // more CTAs than tiles (before the TMEM allocation)
    long long* P = partial + ((size_t)it * ctas_per_item + part) * kStatsPartWords;
    const uint8_t* dgd = dgd_base + s.dgd_off;
    const uint8_t* src = src_base + s.src_off;
    if (s.wiener_win == 7) stats_tc_body<7>(dgd, src, s, part, ctas_per_item, P, smem);
    else if (s.wiener_win == 5) stats_tc_body<5>(dgd, src, s, part, ctas_per_item, P, smem);
    else stats_tc_body<3>(dgd, src, s, part, ctas_per_item, P, smem);
}

// One thread per output element: adds its terms over every partial that was written and applies the mean expansion
// above.  grid = (ceil(2450 / 256), n_items).
__global__ void __launch_bounds__(256)
stats_finalize_kernel(const long long* __restrict__ partial, int parts, const SvtB200StatsItem* __restrict__ items,
                      long long* __restrict__ M_out, long long* __restrict__ H_out) {
    const int it = blockIdx.y, e = blockIdx.x * blockDim.x + threadIdx.x;
    const int win = items[it].wiener_win, w2 = win * win;
    if (e >= w2 * w2 + w2) return;
    const int        used = stats_mma_parts(items[it], parts);
    const long long* P    = partial + (size_t)it * parts * kStatsPartWords;
    auto total = [&](int w) {
        long long v = 0;
        for (int p = 0; p < used; p++) v += P[(size_t)p * kStatsPartWords + w];
        return v;
    };
    const long long n = total(kPartN), v = total(kPartS + w2 / 2) / n, nvv = n * v * v;
    if (e < w2 * w2) {
        const int k = e / w2, l = e - k * w2;
        const long long g = total(kPartG + stats_tri_index(w2, min(k, l), max(k, l)));
        H_out[(size_t)it * 2401 + e] = g - v * (total(kPartS + k) + total(kPartS + l)) + nvv;
    } else {
        const int k = e - w2 * w2;
        M_out[(size_t)it * 49 + k] = total(kPartGx + k) - v * (total(kPartS + k) + total(kPartSx)) + nvv;
    }
}

// scratch of the batch call (per-CTA partials, pixel totals), one per stream: calls enqueued on
// different streams may execute concurrently
struct StatsScratch {
    long long*          acc = nullptr;
    unsigned long long* tot = nullptr;
    size_t              cap = 0;
};
static std::map<cudaStream_t, StatsScratch> g_stats;
static std::mutex g_stats_mu;
static ResetHook g_stats_reset([] { std::lock_guard<std::mutex> lk(g_stats_mu); g_stats.clear(); });

template <typename PIX, int WIN>
static void launch_lag_bulk(const PIX* d_dgd, const PIX* d_src, const SvtB200StatsItem* d_items, int n, int cpi, unsigned long long* acc,
                            cudaStream_t st) {
    constexpr size_t smem = lag_bulk_smem<PIX, WIN>();
    static int attr = -1;
    if (attr != epoch()) {
        if (smem > 48 * 1024)
            B200_CUDA_CHECK(cudaFuncSetAttribute(stats_lag_bulk_kernel<PIX, WIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr = epoch();
    }
    stats_lag_bulk_kernel<PIX, WIN><<<dim3(cpi, n), 256, smem, st>>>(d_dgd, d_src, d_items, acc);
    B200_LAUNCH_CHECK();
}

// 8-bit statistics: stats_mma_kernel writes a partial per CTA with pixel tiles, stats_finalize_kernel combines them
static void launch_stats_mma(const uint8_t* d_dgd, const uint8_t* d_src, const SvtB200StatsItem* d_items, int n, long long* d_M,
                             long long* d_H, long long* d_acc, cudaStream_t st) {
    // CTAs per item: ~6 per SM over the batch (two are resident per SM; the kernel gives each of them a few pixel tiles)
    int cpi = (ctx().sm_count * 6) / (n > 0 ? n : 1);
    if (cpi < 1) cpi = 1;
    if (cpi > kStatsMaxParts) cpi = kStatsMaxParts;
    static int attr = -1;
    if (attr != epoch()) {
        B200_CUDA_CHECK(cudaFuncSetAttribute(stats_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmem));
        attr = epoch();
    }
    stats_mma_kernel<<<n * cpi, kTcThreads, kTcSmem, st>>>(d_dgd, d_src, d_items, cpi, d_acc);
    B200_LAUNCH_CHECK();
    stats_finalize_kernel<<<dim3((2450 + 255) / 256, n), 256, 0, st>>>(d_acc, cpi, d_items, d_M, d_H);
    B200_LAUNCH_CHECK();
}

// Wiener statistics of a batch of units: 8-bit pictures on the tensor cores (stats_mma_kernel), 10 / 12 bit by lag sums
// (wiener_stats_lag.cuh) -- both exact
template <typename PIX>
static void launch_stats(const PIX* d_dgd, const PIX* d_src, const SvtB200StatsItem* d_items, int n, int bd, long long* d_M,
                         long long* d_H, long long* d_acc, unsigned long long* d_tot, cudaStream_t st) {
    if constexpr (sizeof(PIX) == 1) return launch_stats_mma(d_dgd, d_src, d_items, n, d_M, d_H, d_acc, st);
    const int divider = bd == 12 ? 16 : (bd == 10 ? 4 : 1);
    int cpi = (ctx().sm_count * 8) / (n > 0 ? n : 1);  // CTAs per unit: ~8 resident CTAs per SM over the batch
    if (cpi < 1) cpi = 1;
    if (cpi > 64) cpi = 64;
    unsigned long long* acc = reinterpret_cast<unsigned long long*>(d_acc);
    B200_CUDA_CHECK(cudaMemsetAsync(d_tot, 0, (size_t)n * sizeof(unsigned long long), st));
    B200_CUDA_CHECK(cudaMemsetAsync(acc, 0, (size_t)n * kLagItemWords * sizeof(unsigned long long), st));
    stats_sum_kernel<PIX><<<n * kSumParts, 256, 0, st>>>(d_dgd, d_items, d_tot);
    B200_LAUNCH_CHECK();
    // one launch per window size; units of another size leave at once (a batch mixes 7x7 luma with 5x5 chroma units)
    launch_lag_bulk<PIX, 7>(d_dgd, d_src, d_items, n, cpi, acc, st);
    launch_lag_bulk<PIX, 5>(d_dgd, d_src, d_items, n, cpi, acc, st);
    launch_lag_bulk<PIX, 3>(d_dgd, d_src, d_items, n, cpi, acc, st);
    stats_lag_edges_kernel<PIX><<<dim3(kLagEdge, n), 256, 0, st>>>(d_dgd, d_items, acc);
    B200_LAUNCH_CHECK();
    stats_lag_finalize_kernel<PIX><<<dim3((49 * 50 / 2 + 49 + 127) / 128, n), 128, 0, st>>>(d_dgd, d_items, acc, d_tot, divider, d_M, d_H);
    B200_LAUNCH_CHECK();
}

template <typename PIX>
static void stats_t1(int wiener_win, const PIX* dgd, const PIX* src, int h_start, int h_end, int v_start, int v_end, int dgd_stride,
                     int src_stride, int64_t* M, int64_t* H, int bd) {
    require_ready();
    const int half = wiener_win >> 1, win2 = wiener_win * wiener_win;
    const int w = h_end - h_start, h = v_end - v_start;
    const int dw = w + 2 * half, dh = h + 2 * half;
    LaneGuard l;
    size_t o_d = l->alloc((size_t)dw * dh * sizeof(PIX)), o_s = l->alloc((size_t)w * h * sizeof(PIX)), o_it = l->alloc(sizeof(SvtB200StatsItem));
    size_t in_end = l->used;
    size_t o_M = l->alloc(49 * 8), o_H = l->alloc(2401 * 8), o_acc = l->alloc(kStatsItemWords * 8), o_avg = l->alloc(16);
    for (int r = 0; r < dh; r++)
        memcpy(l->h<PIX>(o_d) + (size_t)r * dw, dgd + (ptrdiff_t)(v_start - half + r) * dgd_stride + h_start - half, dw * sizeof(PIX));
    for (int r = 0; r < h; r++) memcpy(l->h<PIX>(o_s) + (size_t)r * w, src + (ptrdiff_t)(v_start + r) * src_stride + h_start, w * sizeof(PIX));
    SvtB200StatsItem* it = l->h<SvtB200StatsItem>(o_it);
    memset(it, 0, sizeof(*it));
    it->dgd_off = (uint64_t)half * dw + half;  // (v_start, h_start) of the packed copy
    it->src_off = 0;
    it->dgd_stride = dw;
    it->src_stride = w;
    it->h_start = 0;
    it->h_end = w;
    it->v_start = 0;
    it->v_end = h;
    it->wiener_win = wiener_win;
    l->h2d(0, in_end);
    launch_stats<PIX>(l->d<PIX>(o_d), l->d<PIX>(o_s), l->d<SvtB200StatsItem>(o_it), 1, bd, l->d<long long>(o_M), l->d<long long>(o_H),
                      l->d<long long>(o_acc), l->d<unsigned long long>(o_avg), l->stream);
    l->d2h(o_M, (o_H + 2401 * 8) - o_M);
    l->sync();
    memcpy(M, l->h<int64_t>(o_M), (size_t)win2 * 8);
    memcpy(H, l->h<int64_t>(o_H), (size_t)win2 * win2 * 8);
}

template <typename PIX>
static void wiener_t1(const PIX* src, ptrdiff_t src_stride, PIX* dst, ptrdiff_t dst_stride, const int16_t* fx, const int16_t* fy, int w,
                      int h, int round0, int round1, int bd, int lbd_rows) {
    require_ready();
    LaneGuard l;
    const int sw = w + 8, sh = h + 7;
    size_t o_s = l->alloc((size_t)sw * sh * sizeof(PIX)), o_u = l->alloc(sizeof(SvtB200WienerUnit));
    size_t in_end = l->used;
    size_t o_d = l->alloc((size_t)w * h * sizeof(PIX));
    for (int r = 0; r < sh; r++) memcpy(l->h<PIX>(o_s) + (size_t)r * sw, src + (ptrdiff_t)(r - 3) * src_stride - 3, sw * sizeof(PIX));
    SvtB200WienerUnit* u = l->h<SvtB200WienerUnit>(o_u);
    memset(u, 0, sizeof(*u));
    u->src_off = (uint64_t)3 * sw + 3;
    u->dst_off = 0;
    u->src_stride = sw;
    u->dst_stride = w;
    u->w = (uint16_t)w;
    u->h = (uint16_t)h;
    memcpy(u->hfilter, fx, 16);
    memcpy(u->vfilter, fy, 16);
    l->h2d(0, in_end);
    wiener_convolve_kernel<PIX><<<1, 256, 0, l->stream>>>(l->d<PIX>(o_s), l->d<PIX>(o_d), l->d<SvtB200WienerUnit>(o_u), 1, bd, round0, round1, lbd_rows);
    B200_LAUNCH_CHECK();
    l->d2h(o_d, (size_t)w * h * sizeof(PIX));
    l->sync();
    for (int r = 0; r < h; r++) memcpy(dst + (ptrdiff_t)r * dst_stride, l->h<PIX>(o_d) + (size_t)r * w, w * sizeof(PIX));
}

}  // namespace b200

using namespace b200;

extern "C" void svt_b200_av1_wiener_convolve_add_src(const uint8_t* src, ptrdiff_t src_stride, uint8_t* dst, ptrdiff_t dst_stride,
                                                     const int16_t* filter_x, const int16_t* filter_y, int32_t w, int32_t h,
                                                     const SvtB200ConvolveParams* conv_params) {
    wiener_t1<uint8_t>(src, src_stride, dst, dst_stride, filter_x, filter_y, w, h, conv_params->round_0, conv_params->round_1, 8, 1);
}
extern "C" void svt_b200_av1_highbd_wiener_convolve_add_src(const uint16_t* src, ptrdiff_t src_stride, uint16_t* dst,
                                                            ptrdiff_t dst_stride, const int16_t* filter_x, const int16_t* filter_y,
                                                            int32_t w, int32_t h, const SvtB200ConvolveParams* conv_params, int32_t bd) {
    wiener_t1<uint16_t>(src, src_stride, dst, dst_stride, filter_x, filter_y, w, h, conv_params->round_0, conv_params->round_1, bd, 0);
}
extern "C" void svt_b200_av1_compute_stats(int32_t wiener_win, const uint8_t* dgd, const uint8_t* src, int32_t h_start, int32_t h_end,
                                           int32_t v_start, int32_t v_end, int32_t dgd_stride, int32_t src_stride, int64_t* M, int64_t* H) {
    stats_t1<uint8_t>(wiener_win, dgd, src, h_start, h_end, v_start, v_end, dgd_stride, src_stride, M, H, 8);
}
extern "C" void svt_b200_av1_compute_stats_highbd(int32_t wiener_win, const uint16_t* dgd, const uint16_t* src, int32_t h_start,
                                                  int32_t h_end, int32_t v_start, int32_t v_end, int32_t dgd_stride, int32_t src_stride,
                                                  int64_t* M, int64_t* H, int32_t bit_depth) {
    stats_t1<uint16_t>(wiener_win, dgd, src, h_start, h_end, v_start, v_end, dgd_stride, src_stride, M, H, bit_depth);
}

extern "C" int svt_b200_wiener_units_dev(const void* d_src, void* d_dst, const SvtB200WienerUnit* d_units, int n_units, int bit_depth,
                                         void* stream) {
    require_ready();
    if (n_units <= 0) return n_units == 0 ? SVT_B200_OK : SVT_B200_ERR_BAD_ARG;
    // get_conv_params_wiener (convolve.h): round_0 = 3 (+2 at 12 bit), round_1 = 2*FILTER_BITS - round_0
    const int round0 = bit_depth == 12 ? 5 : 3, round1 = 14 - round0;
    cudaStream_t st = (cudaStream_t)stream;
    if (bit_depth > 8)
        wiener_convolve_kernel<uint16_t><<<grid_for(n_units, 4), 256, 0, st>>>((const uint16_t*)d_src, (uint16_t*)d_dst, d_units, n_units, bit_depth, round0, round1, 0);
    else
        wiener_convolve_kernel<uint8_t><<<grid_for(n_units, 4), 256, 0, st>>>((const uint8_t*)d_src, (uint8_t*)d_dst, d_units, n_units, 8, round0, round1, 1);
    B200_LAUNCH_CHECK();
    return SVT_B200_OK;
}

extern "C" int svt_b200_compute_stats_batch_dev(const void* d_dgd, const void* d_src, const SvtB200StatsItem* d_items, int n_items,
                                                int bit_depth, int64_t* d_M, int64_t* d_H, void* stream) {
    require_ready();
    if (n_items <= 0) return n_items == 0 ? SVT_B200_OK : SVT_B200_ERR_BAD_ARG;
    std::lock_guard<std::mutex> lk(g_stats_mu);
    StatsScratch& sc = g_stats[(cudaStream_t)stream];
    if ((size_t)n_items > sc.cap) {
        sc.cap = (size_t)n_items * 2;  // new buffers; the old ones live on until shutdown (captured graphs may replay them)
        sc.acc = (long long*)scratch_alloc(sc.cap * kStatsItemWords * 8);
        sc.tot = (unsigned long long*)scratch_alloc(sc.cap * 8);
    }
    if (bit_depth > 8)
        launch_stats<uint16_t>((const uint16_t*)d_dgd, (const uint16_t*)d_src, d_items, n_items, bit_depth, (long long*)d_M, (long long*)d_H,
                               sc.acc, sc.tot, (cudaStream_t)stream);
    else
        launch_stats<uint8_t>((const uint8_t*)d_dgd, (const uint8_t*)d_src, d_items, n_items, 8, (long long*)d_M, (long long*)d_H, sc.acc,
                              sc.tot, (cudaStream_t)stream);
    return SVT_B200_OK;
}
