// knn_tc1.cu -- the fast tcgen05 distance engine: ONE product of IEEE f16 operands per tile (tcgen05.mma kind::f16),
// a wider candidate list and the same exact certificate.
//
// knn_tc.cu reproduces fp32 ranking by arithmetic (3xTF32).  The certificate of refine_kernel makes
// that unnecessary: any approximate score with a known error bound yields the exact 2-NN as long as
//     d2_exact(second) < min_lists(s_kth) + |q|^2 - eps        (otherwise the query is re-scanned)
// holds, and a single product of operands with 11 significant bits has a worst-case error of 2^-10 (|q|^2 + |t|^2) (inputs
// rounded to 11 significant bits, products exact, fp32 accumulation).  f16 meets all three, as tf32 does, at twice the tf32
// rate and half the bytes.  Only columns within twice that error of the running second best are kept (up to 8 per list:
// near-ties overflow 4), which for SURF-like data leaves almost nothing to re-scan, so the kernel issues a fifth of the
// tensor instructions of 3xTF32, each at twice the rate:
//     5 UMMA instructions per 128 x 256 tile at D = 64 (4 + the norm step) instead of 24.
// At that rate the L2 -> shared-memory feed becomes the limiter, so every train tile (32 KB per k chunk) that TMA
// brings in is multiplied against TWO resident query tiles (256 queries), alternating between the
// two TMEM accumulators.  Results are identical to the exact engine by construction.
#include "tc_common.cuh"

#include <cuda_fp16.h>

namespace erp {

constexpr int F_BM = 128;                 // queries per sub-tile (UMMA M)
constexpr int F_SUB = 2;                  // resident query sub-tiles sharing every train tile
constexpr int F_BN = 256;                 // train rows per tile (UMMA N)
constexpr int F_KC = 64;                  // halves per k chunk: one 128-byte swizzle row
constexpr int F_QCH = F_BM * 128;         // 16 KB
constexpr int F_TCH = F_BN * 128;         // 32 KB
constexpr int F_EPI_GROUPS = 2;
constexpr int F_EPI_THREADS = F_EPI_GROUPS * 128;
constexpr int F_THREADS = 128 + F_EPI_THREADS;
constexpr int F_EPI_COLS = F_BN / F_EPI_GROUPS;
constexpr int F_TOPK = 8;
constexpr int F_MAX_SEG = 128 / (F_TOPK * F_EPI_GROUPS);    // up to 8 segments per query pair (refine_kernel: 128 candidate slots)
constexpr int F_AUG_T = F_BN * 32;        // 8 KB: one extra k step (16 halves) per train row, 32-byte swizzle rows
constexpr int F_AUG_Q = F_BM * 32;        // 4 KB: the constant query side of that k step
constexpr int F_BARS = 256;               // mbarriers + TMEM slot
// |s_tc - s_exact| <= 2^-10 (|q|^2 + max|t|^2) in the worst case: both operands are rounded to 11
// significant bits (relative error 2^-11 each, f16 rounds to nearest even), products are exact (11 x 11 bits fit fp32,
// and so do f16 subnormal products), and 2|q||t| <= |q|^2 + |t|^2.
// On top of 2^-10: the second-order rounding term (2^-22 relative = 2^-12 of the budget), the column id packed into the
// three low mantissa bits of a score (<= 7 ulp = 2^-21 relative), and the fp32 accumulation inside the tensor pipe,
// whose rounding mode is not documented: with truncating adds over D + 3 <= 131 terms the worst case is 131 * 2^-24
// of the scale = 0.8 % of 2^-10.  Together < 2 %; 5 % is taken.  refine_kernel reports the deviation it observes
// (0.28 of the bound on the synthetic sets; tests/test_gpu_parity.py holds a worst-case-rounding adversarial set).
// f16 adds two things the relative bound does not cover, both handled without a host round trip:
//   - values f16 cannot hold (|x| >= 65520 after the query's x(-2), or |t|^2 >= 65520 * 2^8 for the norm step): the prep
//     kernel raises misc[5] and refine_kernel re-scans every query of the call exactly;
//   - subnormal f16 operands (|x| < 2^-14) carry an absolute error <= 2^-25 each instead of a relative one, so a product
//     errs by at most 2^-25 (|a~| + |b~|) beyond the relative term, which sums to <= 2^-25 sqrt(D) (2|q| + max|t|) (1 + 2^-10);
//     the norm step adds <= 2^-39.  refine_kernel certifies a query only while 2^-24 sqrt(D) (2|q| + max|t|) + 2^-36 -- twice
//     that -- stays within F_F16_ABS of the scale, 2 % of 2^-10 of the 3 % the budget above leaves.  That holds whenever
//     |q| or max|t| is above ~0.1 (SURF is unit-norm, SIFT far above), so real descriptors never take this path.
constexpr double F_KAPPA = 1.05 / 1024.0;
constexpr double F_F16_ABS = 0.02 / 1024.0;
// instruction descriptor: D fp32, A/B f16 (format 0), both K-major, N = 256, M = 128
constexpr uint32_t F_IDESC = (1u << 4) | ((uint32_t)(F_BN >> 3) << 17) | ((uint32_t)(F_BM >> 4) << 24);
// |t|^2 enters the accumulator through the tensor core, as an extra k step after the k chunks, so the epilogue neither
// loads nor adds it.  Norm step: train row (hi, mid, lo, 0 x 5 | 0 x 8), query row (2^8, 2^-3, 2^-14, 2^15 x 5) in both
// 16-byte halves, so |t|^2 = 2^8 hi + 2^-3 mid + 2^-14 lo (a 33-bit split of the fp32 norm: exact while hi is normal,
// within 2^-39 below).  Padding train rows put 65504 into the five 2^15 slots: 1.07e10, finite, and above any score the
// range guard lets through (|2q| |t| <= 65504 sqrt(128) * 4096 = 3.0e9 plus |t|^2 < 1.7e7)
__host__ __device__ constexpr float f16_norm_scale(int i) { return i == 0 ? 256.0f : i == 1 ? 0.125f : i == 2 ? 1.0f / 16384.0f : 32768.0f; }

// shared memory behind the query chunks and the T ring: the norm operand (two train tiles and the query side), the barriers,
// and the per-row threshold exchange between the two column groups (512 B per sub-tile)
constexpr int F_TAIL = 2 * F_AUG_T + F_AUG_Q + F_BARS + F_SUB * F_BM * 4;
__host__ __device__ constexpr int f_slots(int kch) { return (TC_SMEM_LIMIT - F_SUB * kch * F_QCH - F_TAIL) / F_TCH; }
__host__ __device__ constexpr int f_smem(int kch) { return F_SUB * kch * F_QCH + f_slots(kch) * F_TCH + F_TAIL; }

// one operand of a prep launch: rows x, scaled, rounded to f16 into out (dpad halves per row); norms (+inf padding up to n_pad),
// their maximum, and the 32-byte norm operand rows when aug is given
// LPR lanes own one row (4 elements per lane and pass); a warp covers 32 / LPR rows
struct RoundJob {
    const float* x; int n; float scale; __half* out; float* norm; int n_pad; unsigned* max_bits; __half* aug; int blocks;
};

// f16 of a scaled input; a finite input whose f16 is infinite marks the call for the exact re-scan
__device__ __forceinline__ __half f16_guarded(float x, float scaled, bool& wide)
{
    const __half h = __float2half_rn(scaled);
    wide |= __hisinf(h) != 0 && fabsf(x) <= 3.4028235e38f;
    return h;
}

// both operands of a search in ONE launch: blocks [0, a.blocks) round the queries, the rest the train rows
template <int LPR>
__global__ void __launch_bounds__(256)
round_kernel(const RoundJob a, const RoundJob b, int dim, int dpad, unsigned* wide_flag)
{
    constexpr int RPW = 32 / LPR;
    const bool second = (int)blockIdx.x >= a.blocks;
    const RoundJob& j = second ? b : a;
    const float* __restrict__ x = j.x;
    float* __restrict__ norm = j.norm;
    unsigned* __restrict__ max_bits = j.max_bits;
    const int n = j.n, n_pad = j.n_pad;
    const float scale = j.scale;
    const int lane = threadIdx.x & 31, sub = lane / LPR, l = lane % LPR;
    const int row = (((int)blockIdx.x - (second ? a.blocks : 0)) * 8 + (threadIdx.x >> 5)) * RPW + sub;
    double acc = 0.0;
    bool wide = false;
    if (row < n) {
        for (int k = l * 4; k < dpad; k += LPR * 4) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k < dim) v = *reinterpret_cast<const float4*>(x + (size_t)row * dim + k);
            acc += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
            __half2* o = reinterpret_cast<__half2*>(j.out + (size_t)row * dpad + k);
            o[0] = __halves2half2(f16_guarded(v.x, __fmul_rn(v.x, scale), wide), f16_guarded(v.y, __fmul_rn(v.y, scale), wide));
            o[1] = __halves2half2(f16_guarded(v.z, __fmul_rn(v.z, scale), wide), f16_guarded(v.w, __fmul_rn(v.w, scale), wide));
        }
    }
    if (norm) {
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (l == 0 && row < n_pad) {
            float f = row < n ? (float)acc : INFINITY;
            norm[row] = f;
            if (j.aug) {
                // |t|^2 = 2^8 hi + 2^-3 mid + 2^-14 lo (f16_norm_scale); rows past the end fill the 2^15 slots
                unsigned short h[8] = {0, 0, 0, 0, 0, 0, 0, 0};
                if (row < n) {
                    const __half hi = f16_guarded(f, __fmul_rn(f, 1.0f / f16_norm_scale(0)), wide);
                    const float r1 = __fsub_rn(f, __fmul_rn(__half2float(hi), f16_norm_scale(0)));
                    const __half mid = __float2half_rn(__fmul_rn(r1, 1.0f / f16_norm_scale(1)));
                    const float r2 = __fsub_rn(r1, __fmul_rn(__half2float(mid), f16_norm_scale(1)));
                    const __half lo = __float2half_rn(__fmul_rn(r2, 1.0f / f16_norm_scale(2)));
                    h[0] = __half_as_ushort(hi); h[1] = __half_as_ushort(mid); h[2] = __half_as_ushort(lo);
                } else {
                    for (int i = 3; i < 8; i++) h[i] = 0x7bffu;   // 65504
                }
                uint4* o = reinterpret_cast<uint4*>(j.aug + (size_t)row * 16);
                o[0] = make_uint4(h[0] | (uint32_t)h[1] << 16, h[2] | (uint32_t)h[3] << 16, h[4] | (uint32_t)h[5] << 16, h[6] | (uint32_t)h[7] << 16);
                o[1] = make_uint4(0u, 0u, 0u, 0u);
            }
            // non-negative floats (and +inf, NaN) order like their bit patterns
            // one hot word for the whole array: read it first, the atomic only fires while the maximum still grows
            if (row < n && __float_as_uint(f) > *reinterpret_cast<volatile unsigned*>(max_bits)) atomicMax(max_bits, __float_as_uint(f));
        }
    }
    if (wide) *wide_flag = 1u;
}

static int launch_prep(erp_ctx* ctx, RoundJob a, RoundJob b, int dim, int dpad, unsigned* wide_flag)
{
    // 16 lanes per row for dpad = 64, 32 for dpad = 128
    const int lpr = dpad <= 64 ? 16 : 32;
    const int rows_per_block = 8 * (32 / lpr);
    a.blocks = cdiv(a.n_pad, rows_per_block);
    b.blocks = b.x ? cdiv(b.n_pad, rows_per_block) : 0;
    const int grid = a.blocks + b.blocks;
    if (lpr == 16) round_kernel<16><<<grid, 256, 0, ctx->stream>>>(a, b, dim, dpad, wide_flag);
    else round_kernel<32><<<grid, 256, 0, ctx->stream>>>(a, b, dim, dpad, wide_flag);
    ERP_LAUNCH(ctx, "round_kernel");
    return ERP_OK;
}

struct Tc1Params {
    const float* qn;          // nq query norms |q|^2
    const unsigned* tn_max_bits;
    int32_t* cand_idx;        // nq x lists x F_TOPK, pre-set to -1
    float* cand_s;
    float* cand_thr;          // nq x lists: lower bound of the approximate score of every non-candidate
    int32_t* row_thr;         // nq ordered-int keys (or null): the lowest threshold any segment of the row has published
    int nq, nt;
    int n_qpairs, n_ttiles;   // n_qpairs counts groups of F_SUB query sub-tiles
    int units_per_cta;        // CTA b owns units [b*L, (b+1)*L) of the n_qpairs x n_ttiles grid
    int n_seg;                // candidate lists per query = n_seg x F_EPI_GROUPS
};

// monotone float <-> int key (scores may be negative), so that atomicMin orders thresholds
__device__ __forceinline__ int32_t thr_key(float f) { const int32_t k = __float_as_int(f); return k >= 0 ? k : k ^ 0x7fffffff; }
__device__ __forceinline__ float key_thr(int32_t k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }

template <int KCH>   // KCH k chunks of 128 bytes: dpad = KCH * F_KC halves
__global__ void __launch_bounds__(F_THREADS, 1)
knn2_tc1_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t,
                const __grid_constant__ CUtensorMap map_aug, const Tc1Params p)
{
    constexpr int NS = f_slots(KCH);
    static_assert(NS >= KCH + 1, "T ring must hold one tile plus a chunk of look-ahead");
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* q_smem = smem;                                   // [F_SUB][KCH] chunks
    uint8_t* t_smem = smem + F_SUB * KCH * F_QCH;             // NS slots
    uint8_t* aug_t = t_smem + NS * F_TCH;                     // [2][F_AUG_T] norm operand by train-tile parity, then the query side
    uint8_t* aug_q = aug_t + 2 * F_AUG_T;
    uint64_t* bars = reinterpret_cast<uint64_t*>(aug_q + F_AUG_Q);
    using Pipe = PairPipe<F_SUB, KCH, NS, F_BM, F_BN, F_KC>;
    const Pipe pipe(q_smem, t_smem, bars);
    uint64_t* nfull = bars + Pipe::N_BARS;      // [2] norm operand of a train tile landed
    uint64_t* nempty = nfull + 2;               // [2] ... and read by the MMAs of both sub-tiles
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(nfull + 4);
    static_assert((Pipe::N_BARS + 4) * 8 + 4 <= F_BARS, "barrier block");
    float* thr_sh = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + F_BARS);   // [F_SUB][F_BM] row thresholds
    static_assert(F_SUB * KCH * F_QCH + NS * F_TCH + 2 * F_AUG_T + F_AUG_Q + F_BARS + F_SUB * F_BM * 4 <= f_smem(KCH),
                  "threshold exchange area");
    static_assert(f_smem(KCH) <= TC_SMEM_LIMIT, "shared memory budget");

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    TCC_DECL;
    constexpr int W_ALLOC = F_EPI_THREADS / 32, W_NORM = W_ALLOC + 1, W_TMA = W_ALLOC + 2, W_MMA = W_ALLOC + 3;

    if (warp == W_TMA && lane == 0) { tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_t); tma_prefetch_desc(&map_aug); }
    if (warp == W_MMA && lane == 0) {
        for (int i = 0; i < 2; i++) { mbar_init(&nfull[i], 1); mbar_init(&nempty[i], 1); }
        pipe.init(F_EPI_THREADS / 32);
    }
    // query side of the norm step: the same 8 halves in both 16-byte halves of every row, which the swizzle cannot change
    for (int i = threadIdx.x; i < F_AUG_Q / 2; i += F_THREADS)
        reinterpret_cast<__half*>(aug_q)[i] = __float2half_rn(f16_norm_scale(i & 7));
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const uint32_t tmem_base = tmem_alloc(warp == W_ALLOC, tmem_slot);

    // the four feeder warps need few registers; the eight epilogue warps take them over (4 chunks of 32 accumulator columns in flight)
    if (warp >= W_ALLOC) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
    if (warp == W_TMA) {
        // ================================================================ TMA producer
        if (lane == 0) pipe.produce(&map_q, &map_t, SegIter(p.n_qpairs, p.n_ttiles, p.units_per_cta, blockIdx.x));
    } else if (warp == W_MMA) {
        // ================================================================ MMA issuer
        if (lane == 0) {
            const uint64_t aq_desc = smem_desc_sw32(smem_u32(aug_q));
            pipe.issue(tmem_base, SegIter(p.n_qpairs, p.n_ttiles, p.units_per_cta, blockIdx.x),
                       [](uint32_t d_tmem, uint32_t q, int c, uint32_t b) { mma_chunk<tc_mma_f16>(d_tmem, q + c * F_QCH, b, F_IDESC, c != 0); },
                       [&](int sub, uint32_t tt_n, uint32_t d_tmem) {
                           // the norm step
                           const uint32_t nb = tt_n & 1;
                           if (sub == 0) mbar_wait(&nfull[nb], (tt_n >> 1) & 1);
                           tc_fence_after();
                           tc_mma_f16(d_tmem, aq_desc, smem_desc_sw32(smem_u32(aug_t + nb * F_AUG_T)), F_IDESC, 1);
                           if (sub == F_SUB - 1) tc_commit(&nempty[nb]);
                       });
        }
    } else if (warp == W_NORM) {
        // ================================================================ norm operand producer (one TMA load per train tile)
        if (lane == 0) {
            uint32_t tt_n = 0;
            SegIter it(p.n_qpairs, p.n_ttiles, p.units_per_cta, blockIdx.x);
            int qp, t0, t1, seg;
            while (it.next(qp, t0, t1, seg)) {
                for (int tt = t0; tt < t1; tt++, tt_n++) {
                    const uint32_t nb = tt_n & 1;
                    mbar_wait(&nempty[nb], ((tt_n >> 1) & 1) ^ 1);
                    mbar_expect_tx(&nfull[nb], F_AUG_T);
                    tma_load_2d(&map_aug, &nfull[nb], aug_t + nb * F_AUG_T, 0, tt * F_BN);
                }
            }
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;" ::: "memory");
        // ================================================================ epilogue (2 column groups x 4 lane quarters)
        const int ew = warp & 3, cg = warp >> 2;
        const int row = ew * 32 + lane;
        uint32_t tile_n = 0;
        SegIter it(p.n_qpairs, p.n_ttiles, p.units_per_cta, blockIdx.x);
        int qp, t0, t1, seg;
        while (it.next(qp, t0, t1, seg)) {
            float bs[F_SUB][F_TOPK];
            int bi[F_SUB][F_TOPK];
#pragma unroll
            for (int sub = 0; sub < F_SUB; sub++)
#pragma unroll
                for (int j = 0; j < F_TOPK; j++) { bs[sub][j] = INFINITY; bi[sub][j] = -1; }
            float slack[F_SUB];
#pragma unroll
            for (int sub = 0; sub < F_SUB; sub++) {
                const int qrow = (qp * F_SUB + sub) * F_BM + row;
                slack[sub] = slack_of(qrow < p.nq ? p.qn[qrow] : 0.f, __uint_as_float(*p.tn_max_bits), (float)F_KAPPA);
            }
            float floor_thr[F_SUB];
#pragma unroll
            for (int sub = 0; sub < F_SUB; sub++) floor_thr[sub] = INFINITY;
            // A query row cut into several segments is scanned by several CTAs at once, each starting cold.  Any threshold
            // one of them has reached (second best so far + slack) bounds the row's exact two nearest for ALL of them, so
            // the segments publish theirs (atomicMin on an ordered key) and fold the others' in every few tiles: the row
            // then warms up once, not once per segment.  Racy on purpose: every published value is a valid bound, and
            // floor_thr -- the lowest threshold ever in force -- is what the list's certificate bound is built from.
            const bool seed = p.row_thr != nullptr;
            float published[F_SUB];
#pragma unroll
            for (int sub = 0; sub < F_SUB; sub++) published[sub] = INFINITY;
            // every epilogue warp has left the previous query rows before their thresholds are replaced
            asm volatile("bar.sync 1, %0;" ::"n"(F_EPI_THREADS) : "memory");
#pragma unroll
            for (int sub = 0; sub < F_SUB; sub++) {
                const int qrow = (qp * F_SUB + sub) * F_BM + row;
                float g = INFINITY;
                if (seed && qrow < p.nq) g = key_thr(*reinterpret_cast<volatile int32_t*>(p.row_thr + qrow));
                thr_sh[sub * F_BM + row] = g;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(F_EPI_THREADS) : "memory");
            for (int tt = t0; tt < t1; tt++) {
                // every fourth tile: fetch the row's published bound now, use it after this tile's scan
                const bool sync_thr = seed && ((tt - t0) & 3) == 3;
                int32_t fetched[F_SUB];
                if (sync_thr) {
#pragma unroll
                    for (int sub = 0; sub < F_SUB; sub++) {
                        const int qrow = (qp * F_SUB + sub) * F_BM + row;
                        fetched[sub] = qrow < p.nq ? *reinterpret_cast<volatile int32_t*>(p.row_thr + qrow) : 0x7f7f7f7f;
                    }
                }
                const int colbase = tt * F_BN + cg * F_EPI_COLS;
#pragma unroll
                for (int sub = 0; sub < F_SUB; sub++, tile_n++) {
                    const uint32_t acc = tile_n & 1;
                    TCC_CLOCK(c0);
                    mbar_wait(&pipe.tfull[acc], (tile_n >> 1) & 1);
                    TCC_CLOCK(c1);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + acc * F_BN + cg * F_EPI_COLS;
                    // all four chunks of this warp's share in registers at once: the epilogue warps hold 224 (setmaxnreg above)
                    static_assert(F_EPI_COLS == 128, "four chunks of 32 columns per warp and tile");
                    uint32_t va[32], vb[32], vc[32], vd[32];
                    pipe.drain(taddr, acc, va, vb, vc, vd);
                    scan_chunk_lean(va, colbase, slack[sub], bs[sub], bi[sub], thr_sh + sub * F_BM + row, floor_thr[sub]);
                    scan_chunk_lean(vb, colbase + 32, slack[sub], bs[sub], bi[sub], thr_sh + sub * F_BM + row, floor_thr[sub]);
                    scan_chunk_lean(vc, colbase + 64, slack[sub], bs[sub], bi[sub], thr_sh + sub * F_BM + row, floor_thr[sub]);
                    scan_chunk_lean(vd, colbase + 96, slack[sub], bs[sub], bi[sub], thr_sh + sub * F_BM + row, floor_thr[sub]);
                    TCC_ADD(0, c1 - c0); TCC_ADD(1, clock64() - c1); TCC_ADD(2, 1);
                }
                if (sync_thr) {
#pragma unroll
                    for (int sub = 0; sub < F_SUB; sub++) {
                        const int qrow = (qp * F_SUB + sub) * F_BM + row;
                        if (qrow >= p.nq) continue;
                        const float mine = floor_thr[sub];
                        if (mine < published[sub]) { atomicMin(p.row_thr + qrow, thr_key(mine)); published[sub] = mine; }
                        const float g = key_thr(fetched[sub]);
                        volatile float* rt = thr_sh + sub * F_BM + row;
                        if (g < *rt) *rt = g;
                    }
                }
            }
#pragma unroll
            for (int sub = 0; sub < F_SUB; sub++) {
                const int qg = (qp * F_SUB + sub) * F_BM + row;
                if (seed && qg < p.nq && floor_thr[sub] < published[sub]) atomicMin(p.row_thr + qg, thr_key(floor_thr[sub]));
                if (qg < p.nq) {
                    const size_t l = ((size_t)qg * p.n_seg + seg) * F_EPI_GROUPS + cg;
#pragma unroll
                    for (int j = 0; j < F_TOPK; j += 4) {
                        *reinterpret_cast<int4*>(p.cand_idx + l * F_TOPK + j) = make_int4(bi[sub][j], bi[sub][j + 1], bi[sub][j + 2], bi[sub][j + 3]);
                        *reinterpret_cast<float4*>(p.cand_s + l * F_TOPK + j) = make_float4(bs[sub][j], bs[sub][j + 1], bs[sub][j + 2], bs[sub][j + 3]);
                    }
                    p.cand_thr[l] = fminf(floor_thr[sub], __fadd_rn(bs[sub][1], slack[sub]));
                }
            }
        }
    }

    TCC_FLUSH();
    tmem_free(warp == W_ALLOC, tmem_base);
}

#if ERP_TC_COUNTERS == 2
__global__ void dbg_print_kernel()
{
    printf("warp-events (first lane) steady %llu, %.0f clk each; warm-up %llu, %.0f clk each\n", erp_evt[1], (double)erp_evt[0] / erp_evt[1], erp_evt[3], (double)erp_evt[2] / erp_evt[3]);
    printf("lane-events %llu groups %llu inserts %llu\n", erp_evt[4], erp_evt[5], erp_evt[6]);
    for (int i = 0; i < 8; i++) erp_evt[i] = 0;
}
#endif
#if ERP_TC_COUNTERS == 1
__global__ void dbg_print_kernel()
{
    printf("epi: wait_tfull %.0f scan %.0f per warp-tile (%llu warp-tiles) | mma: wait_tempty %.0f wait_full(sum over chunks) %.0f per tile (%llu tiles)\n",
           (double)erp_clk[0] / erp_clk[2], (double)erp_clk[1] / erp_clk[2], erp_clk[2], (double)erp_clk[3] / erp_clk[4], (double)erp_clk[5] / erp_clk[4], erp_clk[4]);
    for (int i = 0; i < 8; i++) erp_clk[i] = 0;
}
#endif
int knn2_tc1(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
             int32_t* d_idx2, float* d_dist2, double* d_d2)
{
    if (!knn2_tc_supported(nq, nt, dim)) { set_error("tcgen05 engine: unsupported shape nq=%d nt=%d dim=%d", nq, nt, dim); return ERP_E_DIM; }
    const int kch = cdiv(dim, F_KC), dpad = kch * F_KC;     // dim <= 128: one or two k chunks
    const int n_qpairs = cdiv(nq, F_BM * F_SUB), n_ttiles = cdiv(nt, F_BN);
    const StreamK plan = stream_k_plan(n_qpairs, n_ttiles, ctx->sm_count, F_MAX_SEG);
    const int n_seg = plan.n_seg, n_lists = n_seg * F_EPI_GROUPS;

    int st = ERP_OK;
    __half* qs = ctx->scratch<__half>(S_TC_Q, (size_t)nq * dpad, &st);
    __half* ts = ctx->scratch<__half>(S_TC_T, (size_t)nt * dpad, &st);
    float* tn = ctx->scratch<float>(S_TC_TN, (size_t)n_ttiles * F_BN * 9, &st);      // norms, then the 32-byte norm operand rows
    int32_t* cand = ctx->scratch<int32_t>(S_TC_CAND, (size_t)nq * n_lists * (F_TOPK * 2 + 1), &st);
    float* qn = ctx->scratch<float>(S_TC_QN, (size_t)nq + 8, &st);
    int32_t* list = ctx->scratch<int32_t>(S_TC_LIST, (size_t)nq + 8, &st);
    int32_t* misc = ctx->scratch<int32_t>(S_TC_MISC, 8, &st);
    // rows cut into segments exchange their thresholds (see the kernel): 12.5k x 100k (one rank of an 8-way split, 5 segments
    // per row) 0.308 -> 0.260 ms, 25k x 100k 0.519 -> 0.474, 100k x 100k (2 segments) 1.759 -> 1.731
    static const int seed_from = [] { const char* e = getenv("ERP_B200_SEED_SEGS"); return e ? atoi(e) : 2; }();     // experiments: 99 = never
    int32_t* row_thr = n_seg >= seed_from ? ctx->scratch<int32_t>(S_TC_ROWTHR, (size_t)nq + 8, &st) : nullptr;
    ERP_TRY(st);
    if (row_thr) ERP_CUDA(cudaMemsetAsync(row_thr, 0x7f, sizeof(int32_t) * (size_t)nq, ctx->stream));
    float* cand_s = reinterpret_cast<float*>(cand + (size_t)nq * n_lists * F_TOPK);
    float* cand_thr = cand_s + (size_t)nq * n_lists * F_TOPK;
    ERP_CUDA(cudaMemsetAsync(cand_thr, 0x7f, (size_t)nq * n_lists * sizeof(float), ctx->stream));              // ~3.4e38: "unbounded"
    ERP_TRY(tc_misc_begin(ctx, misc));
    ERP_CUDA(cudaMemsetAsync(cand, 0xFF, (size_t)nq * n_lists * F_TOPK * sizeof(int32_t), ctx->stream));

    __half* aug = reinterpret_cast<__half*>(tn + (size_t)n_ttiles * F_BN);
    RoundJob jq = {d_q, nq, -2.0f, qs, qn, nq, reinterpret_cast<unsigned*>(misc + 3), nullptr, 0};
    RoundJob jt = {ctx->tc_chunk == 0 ? d_t : nullptr, nt, 1.0f, ts, tn, n_ttiles * F_BN, reinterpret_cast<unsigned*>(misc + 1), aug, 0};
    ERP_TRY(launch_prep(ctx, jq, jt, dim, dpad, reinterpret_cast<unsigned*>(misc + 5)));

    CUtensorMap mq, mt, ma;
    ERP_TRY(make_map(&mq, qs, nq, dpad, F_BM, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2));
    ERP_TRY(make_map(&mt, ts, nt, dpad, F_BN, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2));
    ERP_TRY(make_map(&ma, aug, n_ttiles * F_BN, 16, F_BN, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, true));     // 16 halves: one 32-byte row per train row
    Tc1Params p;
    p.nq = nq; p.nt = nt; p.n_qpairs = n_qpairs; p.n_ttiles = n_ttiles; p.units_per_cta = plan.units_per_cta; p.n_seg = n_seg;
    p.cand_idx = cand; p.cand_s = cand_s; p.cand_thr = cand_thr; p.qn = qn;
    p.tn_max_bits = reinterpret_cast<const unsigned*>(misc + 1);
    p.row_thr = row_thr;

    if (ctx->tc_chunk == 0) ERP_CUDA(record_timing(ctx, ctx->ev_k0));
    if (kch == 1) ERP_TRY(launch_tc_kernel<knn2_tc1_kernel<1>>(ctx, "knn2_tc1_kernel", plan.grid, F_THREADS, f_smem(1), mq, mt, ma, p));
    else ERP_TRY(launch_tc_kernel<knn2_tc1_kernel<2>>(ctx, "knn2_tc1_kernel", plan.grid, F_THREADS, f_smem(2), mq, mt, ma, p));
#if ERP_TC_COUNTERS
    dbg_print_kernel<<<1, 1, 0, ctx->stream>>>();
    cudaStreamSynchronize(ctx->stream);
#endif
    ERP_CUDA(record_timing(ctx, ctx->ev_k1));

    ERP_TRY(refine_launch(ctx, d_q, nq, d_t, nt, dim, n_lists, F_TOPK, F_KAPPA, F_F16_ABS, cand, cand_s, cand_thr,
                          reinterpret_cast<unsigned*>(misc),
                          d_idx2, d_dist2, d_d2, list));
    ERP_TRY(knn2_exact_rescan(ctx, d_q, nq, d_t, nt, dim, list, misc, nq, d_idx2, d_dist2, d_d2));
    ERP_TRY(tc_misc_end(ctx, misc));

    set_knn_stats(ctx, ERP_ENGINE_TCGEN05_1X, false, n_seg, plan.units_per_cta, plan.grid, misc);
    return ERP_OK;
}

} // namespace erp
