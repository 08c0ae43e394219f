// knn_tc.cu -- the tcgen05 distance engine: 3xTF32 GEMM-form tiles with a fused top-4 epilogue,
// followed by an exact fp64 refine that CERTIFIES each query or sends it to the exact re-scan.
//
// Replaces cv::DescriptorMatcher::knnMatch(k=2) of /root/reference/src/feature_matcher.cpp:45 in its
// exact-L2 limit (SURVEY D1).  Pipeline, all on ctx->stream, no host synchronisation:
//
//   split_kernel (x2)   fp32 rows -> TF32 pairs (hi = rna_tf32(v), lo = rna_tf32(v - hi)), interleaved in
//                       32-float chunks [hi_0 | lo_0 | hi_1 | lo_1 | ...], query rows pre-scaled by -2
//                       (exact), train norms |t|^2, max norm
//   knn2_tc_kernel      persistent (one CTA per SM owns a contiguous range of (query tile, train tile)
//                       units, stream-K style, so SMs finish together), warp specialised, on the query-pair
//                       pipeline of tc_common.cuh (PairPipe, one query sub-tile of 2 x KCH chunks):
//                       TMA (128B-swizzled K-major boxes) -> smem ring, a train tile's chunks in row order
//                       -> tcgen05.mma kind::tf32, three products per 32-wide k chunk
//                       (lo*hi + hi*hi + hi*lo) accumulated in a TMEM tile of 128 queries x 256 train
//                       rows, double buffered (2 x 256 columns) so the epilogue of tile i overlaps
//                       the MMAs of tile i+1.  Epilogue: tcgen05.ld 32x32b (one query row per
//                       thread), s = acc + |t|^2, running top-4 per row in registers.  The distance
//                       matrix never leaves the SM.
//   refine_kernel       exact fp64 direct-form distance (the oracle's fma chain) of the candidates,
//                       lexicographic (d2, index) top-2, and the certificate
//                           d2_exact(second) < min_split(s_4th) + |q|^2 - eps
//                       (every non-candidate has approximate score >= s_4th, so its exact distance
//                       is >= s_4th + |q|^2 - eps).  Uncertified queries go to a list.
//   re-scan             the listed queries through the exact fp64 kernel (knn_exact.cu), T-split for
//                       short lists.  Results are therefore identical to ERP_ENGINE_EXACT_SIMT.
#include "tc_common.cuh"

namespace erp {

// ------------------------------------------------------------------------------------------
// tile configuration
// ------------------------------------------------------------------------------------------
constexpr int BM = 128;                 // queries per tile  (UMMA M, TMEM lanes)
constexpr int BN = 256;                 // train rows per tile (UMMA N, TMEM columns per accumulator)
constexpr int KC = 32;                  // floats per k chunk: one 128-byte swizzle atom
constexpr int Q_CHUNK_BYTES = BM * KC * 4;   // 16 KB
constexpr int T_CHUNK_BYTES = BN * KC * 4;   // 32 KB
constexpr int EPI_GROUPS = 2;           // column groups per tile: 2 x 4 epilogue warps, two per scheduler
constexpr int EPI_THREADS = EPI_GROUPS * 128;
constexpr int TC_THREADS = 128 + EPI_THREADS;   // warps 0..7 epilogue, then TMEM alloc, |t|^2 loads, TMA, MMA
constexpr int EPI_COLS = BN / EPI_GROUPS;       // columns of a tile each epilogue thread scans
constexpr int TOPK = 4;
constexpr int MAX_SEG = 64 / (TOPK * EPI_GROUPS);     // segments per query tile: refine_kernel holds <= 64 candidates
constexpr int SMEM_LIMIT = TC_SMEM_LIMIT;       // the budget of n_slots (tests/test_gpu_pipeline_plans.py reads the formula by name)
constexpr int SMEM_TAIL = 2 * BN * 4 + 256;     // |t|^2 of two tiles + mbarriers + the TMEM base address
// certificate slack: |s_tc - s_exact| <= KAPPA * (|q|^2 + max|t|^2).  3xTF32 drops lo*lo (2^-22),
// rounds lo to tf32 (2^-23) and accumulates 3*D/8 partial sums in fp32 (<= 2^-18 for D = 128);
// 2^-14 leaves a factor > 8.  refine_kernel reports the largest deviation it observes.
constexpr double KAPPA = 1.0 / 16384.0;

__host__ __device__ constexpr int n_slots(int kch) { return (SMEM_LIMIT - 2 * kch * Q_CHUNK_BYTES - SMEM_TAIL) / T_CHUNK_BYTES; }
__host__ __device__ constexpr int tc_smem(int kch) { return 2 * kch * Q_CHUNK_BYTES + n_slots(kch) * T_CHUNK_BYTES + SMEM_TAIL; }

constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// ------------------------------------------------------------------------------------------
// prep: fp32 rows -> hi and lo (dpad each, interleaved by k chunk), norms
// ------------------------------------------------------------------------------------------

// one warp per row.  out: n x (2*dpad), chunk c of hi at 2c * KC, of lo at (2c + 1) * KC.  norm (optional): n_pad floats, rows >= n get +inf.
// LPR lanes own one row (4 floats per lane and pass); a warp covers 32 / LPR rows
template <int LPR>
__global__ void __launch_bounds__(256)
split_kernel(const float* __restrict__ x, int n, int dim, int dpad, float scale,
             float* __restrict__ out, float* __restrict__ norm, int n_pad, unsigned* __restrict__ max_bits)
{
    constexpr int RPW = 32 / LPR;
    const int lane = threadIdx.x & 31, sub = lane / LPR, l = lane % LPR;
    const int row = (blockIdx.x * 8 + (threadIdx.x >> 5)) * RPW + sub;
    double acc = 0.0;
    if (row < n) {
        for (int k = l * 4; k < dpad; k += LPR * 4) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (k < dim) v = *reinterpret_cast<const float4*>(x + (size_t)row * dim + k);
            acc += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
            float4 s = make_float4(__fmul_rn(v.x, scale), __fmul_rn(v.y, scale), __fmul_rn(v.z, scale), __fmul_rn(v.w, scale));
            float4 hi = make_float4(tf32_rna(s.x), tf32_rna(s.y), tf32_rna(s.z), tf32_rna(s.w));
            float4 lo = make_float4(tf32_rna(__fsub_rn(s.x, hi.x)), tf32_rna(__fsub_rn(s.y, hi.y)),
                                    tf32_rna(__fsub_rn(s.z, hi.z)), tf32_rna(__fsub_rn(s.w, hi.w)));
            float* o = out + (size_t)row * 2 * dpad + (k & ~(KC - 1)) + k;
            *reinterpret_cast<float4*>(o) = hi;
            *reinterpret_cast<float4*>(o + KC) = lo;
        }
    }
    if (norm) {
#pragma unroll
        for (int o = LPR / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (l == 0 && row < n_pad) {
            float f = row < n ? (float)acc : INFINITY;
            norm[row] = f;
            // non-negative floats (and +inf, NaN) order like their bit patterns
            // one hot word for the whole array: read it first, the atomic only fires while the maximum still grows
            if (row < n && __float_as_uint(f) > *reinterpret_cast<volatile unsigned*>(max_bits)) atomicMax(max_bits, __float_as_uint(f));
        }
    }
}

static int launch_prep(erp_ctx* ctx, const float* x, int n, int dim, int dpad, float scale, float* out, float* norm, int n_pad,
                       unsigned* max_bits)
{
    // 8 / 16 / 32 lanes per row for dpad = 32 / 64 / (96, 128)
    const int lpr = dpad <= 32 ? 8 : dpad <= 64 ? 16 : 32;
    const int rows_per_block = 8 * (32 / lpr);
    const int grid = cdiv(n_pad, rows_per_block);
    if (lpr == 8) split_kernel<8><<<grid, 256, 0, ctx->stream>>>(x, n, dim, dpad, scale, out, norm, n_pad, max_bits);
    else if (lpr == 16) split_kernel<16><<<grid, 256, 0, ctx->stream>>>(x, n, dim, dpad, scale, out, norm, n_pad, max_bits);
    else split_kernel<32><<<grid, 256, 0, ctx->stream>>>(x, n, dim, dpad, scale, out, norm, n_pad, max_bits);
    ERP_LAUNCH(ctx, "split_kernel");
    return ERP_OK;
}

// ---- running top-4 of one query row -----------------------------------------------------------
// A column is a candidate iff its approximate score is below
//     min( 4th best so far,  2nd best so far + slack )      (slack_of, tc_common.cuh).
// Columns above "2nd best + 2 eps" can never be one of the exact two nearest neighbours, so they need not be kept: the
// rare insert path then runs ~2 ln(n) times per row instead of 4 ln(n) or 8 ln(n), and the list's certificate bound is
// that same minimum (both terms only decrease while the scan proceeds).
__device__ __forceinline__ void top4_insert(float s, int idx, float (&bs)[4], int (&bi)[4])
{
    // strict <: equal scores keep the earlier (lower) train index
    if (s < bs[2]) {
        bs[3] = bs[2]; bi[3] = bi[2];
        if (s < bs[1]) {
            bs[2] = bs[1]; bi[2] = bi[1];
            if (s < bs[0]) { bs[1] = bs[0]; bi[1] = bi[0]; bs[0] = s; bi[0] = idx; }
            else { bs[1] = s; bi[1] = idx; }
        } else { bs[2] = s; bi[2] = idx; }
    } else { bs[3] = s; bi[3] = idx; }
}

// 32 accumulator columns of one query row.  Common case: s = acc + |t|^2 (32 independent adds), a min
// tree and ONE warp-uniform threshold test.  Rare case: only the groups of 8 columns that some lane
// needs are re-read from TMEM in a rolled loop, and only the columns below the threshold are visited
// -- the insert cascade exists once per call site, which keeps the loop inside the instruction cache
// (fully unrolled it was 60 KB and 3x slower).  Re-computed scores are bit-identical to the first pass.
__device__ __forceinline__ void scan_chunk(const uint32_t (&v)[32], uint32_t taddr, const float4* __restrict__ tn4, int col0,
                                           float slack, float (&bs)[4], int (&bi)[4])
{
    float gm[4];
#pragma unroll
    for (int g = 0; g < 4; g++) {
        float4 na = tn4[g * 2], nb = tn4[g * 2 + 1];
        float s0 = __fadd_rn(__uint_as_float(v[g * 8 + 0]), na.x), s1 = __fadd_rn(__uint_as_float(v[g * 8 + 1]), na.y);
        float s2 = __fadd_rn(__uint_as_float(v[g * 8 + 2]), na.z), s3 = __fadd_rn(__uint_as_float(v[g * 8 + 3]), na.w);
        float s4 = __fadd_rn(__uint_as_float(v[g * 8 + 4]), nb.x), s5 = __fadd_rn(__uint_as_float(v[g * 8 + 5]), nb.y);
        float s6 = __fadd_rn(__uint_as_float(v[g * 8 + 6]), nb.z), s7 = __fadd_rn(__uint_as_float(v[g * 8 + 7]), nb.w);
        gm[g] = fminf(fminf(fminf(s0, s1), fminf(s2, s3)), fminf(fminf(s4, s5), fminf(s6, s7)));
    }
    const float thr = fminf(bs[3], __fadd_rn(bs[1], slack));
    const unsigned mine = (gm[0] < thr ? 1u : 0u) | (gm[1] < thr ? 2u : 0u) | (gm[2] < thr ? 4u : 0u) | (gm[3] < thr ? 8u : 0u);
    unsigned need = __reduce_or_sync(0xffffffffu, mine);
    while (need) {                                  // warp-uniform
        const int g = __ffs(need) - 1;
        need &= need - 1;
        uint32_t w[8];
        tc_ld8(taddr + g * 8, w);
        tc_wait_ld8(w);
        const float4 na = tn4[g * 2], nb = tn4[g * 2 + 1];
        if ((mine >> g) & 1u) {
            float e[8];
            e[0] = __fadd_rn(__uint_as_float(w[0]), na.x); e[1] = __fadd_rn(__uint_as_float(w[1]), na.y);
            e[2] = __fadd_rn(__uint_as_float(w[2]), na.z); e[3] = __fadd_rn(__uint_as_float(w[3]), na.w);
            e[4] = __fadd_rn(__uint_as_float(w[4]), nb.x); e[5] = __fadd_rn(__uint_as_float(w[5]), nb.y);
            e[6] = __fadd_rn(__uint_as_float(w[6]), nb.z); e[7] = __fadd_rn(__uint_as_float(w[7]), nb.w);
            unsigned m = (e[0] < thr ? 1u : 0u) | (e[1] < thr ? 2u : 0u) | (e[2] < thr ? 4u : 0u) | (e[3] < thr ? 8u : 0u) |
                         (e[4] < thr ? 16u : 0u) | (e[5] < thr ? 32u : 0u) | (e[6] < thr ? 64u : 0u) | (e[7] < thr ? 128u : 0u);
            while (m) {                             // usually a single column
                const int j = __ffs(m) - 1;
                m &= m - 1;
                const float x = j == 0 ? e[0] : j == 1 ? e[1] : j == 2 ? e[2] : j == 3 ? e[3] : j == 4 ? e[4] : j == 5 ? e[5] : j == 6 ? e[6] : e[7];
                if (x < fminf(bs[3], __fadd_rn(bs[1], slack))) top4_insert(x, col0 + g * 8 + j, bs, bi);
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// the distance kernel
// ------------------------------------------------------------------------------------------
struct TcParams {
    int nq, nt;
    int n_qtiles, n_ttiles;
    int units_per_cta;        // L: CTA b owns units [b*L, (b+1)*L) of the n_qtiles x n_ttiles grid (query tile major)
    int n_seg;                // candidate lists per query = n_seg x EPI_GROUPS
    const float* tn;          // n_ttiles * BN norms (+inf padded)
    const float* qn;          // nq query norms |q|^2
    const unsigned* tn_max_bits;
    float* cand_thr;          // nq x lists: lower bound of the approximate score of every non-candidate of the list
    int32_t* cand_idx;        // nq x (n_seg * EPI_GROUPS) x TOPK, pre-set to -1
    float* cand_s;            // same shape: approximate scores, ascending
};

template <int KCH>   // k chunks of 32 floats per half (hi or lo): dpad = 32 * KCH
__global__ void __launch_bounds__(TC_THREADS, 1)
knn2_tc_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t, const TcParams p)
{
    constexpr int NS = n_slots(KCH);
    static_assert(NS >= 2, "T ring too small");
    static_assert(tc_smem(KCH) <= SMEM_LIMIT, "shared memory budget");
    extern __shared__ __align__(1024) uint8_t smem[];
    // the 128B swizzle atoms need a 1024-byte aligned base; the budget has no room for a round-up
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* t_smem = smem + 2 * KCH * Q_CHUNK_BYTES;         // NS slots
    float* tn_smem = reinterpret_cast<float*>(t_smem + NS * T_CHUNK_BYTES);   // [2][BN], follows the accumulator parity
    uint64_t* bars = reinterpret_cast<uint64_t*>(tn_smem + 2 * BN);
    // one query sub-tile of 2*KCH chunks hi_0, lo_0, hi_1, ... (the split rows' order), which is also the order in which a
    // train tile's chunks pass the ring
    using Pipe = PairPipe<1, 2 * KCH, NS, BM, BN, KC>;
    const Pipe pipe(smem, t_smem, bars);
    uint64_t* nfull = bars + Pipe::N_BARS;      // [2] |t|^2 of the tile landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(nfull + 2);
    static_assert((Pipe::N_BARS + 2) * 8 + 4 <= SMEM_TAIL - 2 * BN * 4, "barrier block");

    // the scheduler favours the highest warp id among eligible warps: the single-thread feeders
    // (TMA, MMA) sit on top so that the epilogue warps never delay them
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int W_ALLOC = EPI_THREADS / 32, W_NORM = W_ALLOC + 1, W_TMA = W_ALLOC + 2, W_MMA = W_ALLOC + 3;

    if (warp == W_TMA && lane == 0) {
        tma_prefetch_desc(&map_q);
        tma_prefetch_desc(&map_t);
    }
    if (warp == W_MMA && lane == 0) {
        for (int i = 0; i < 2; i++) mbar_init(&nfull[i], 1);
        pipe.init(EPI_THREADS / 32);
    }
    const uint32_t tmem_base = tmem_alloc(warp == W_ALLOC, tmem_slot);

    if (warp == W_TMA) {
        // ================================================================ TMA producer
        if (lane == 0) pipe.produce(&map_q, &map_t, SegIter(p.n_qtiles, p.n_ttiles, p.units_per_cta, blockIdx.x));
    } else if (warp == W_MMA) {
        // ================================================================ MMA issuer
        if (lane == 0)
            pipe.issue(tmem_base, SegIter(p.n_qtiles, p.n_ttiles, p.units_per_cta, blockIdx.x),
                       [](uint32_t d_tmem, uint32_t q, int c, uint32_t b) {
                           // ring chunk c is T hi_j (c = 2j: lo*hi, then hi*hi) or T lo_j (c = 2j + 1: hi*lo)
                           const uint32_t q_hi = q + (c & ~1) * Q_CHUNK_BYTES, q_lo = q_hi + Q_CHUNK_BYTES;
                           if ((c & 1) == 0) mma_chunk<tc_mma_tf32>(d_tmem, q_lo, b, IDESC, c != 0);
                           mma_chunk<tc_mma_tf32>(d_tmem, q_hi, b, IDESC, true);
                       },
                       [](int, uint32_t, uint32_t) {});
    } else if (warp == W_NORM) {
        // ================================================================ |t|^2 producer
        // one bulk copy of 1 KB per tile into the buffer of the accumulator parity; it may be
        // overwritten once the epilogue has drained that accumulator (the MMA warp's condition too)
        if (lane == 0) {
            uint32_t tile_n = 0;
            SegIter it(p.n_qtiles, p.n_ttiles, p.units_per_cta, blockIdx.x);
            int qtile, t_begin, t_end, seg;
            while (it.next(qtile, t_begin, t_end, seg)) {
                for (int tt = t_begin; tt < t_end; tt++, tile_n++) {
                    const uint32_t acc = tile_n & 1;
                    mbar_wait(&pipe.tempty[acc], ((tile_n >> 1) & 1) ^ 1);
                    mbar_expect_tx(&nfull[acc], BN * 4);
                    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                 ::"r"(smem_u32(tn_smem + acc * BN)), "l"(p.tn + (size_t)tt * BN), "r"(BN * 4), "r"(smem_u32(&nfull[acc]))
                                 : "memory");
                }
            }
        }
    } else if (warp < W_ALLOC) {
        // ================================================================ epilogue (EPI_GROUPS x 4 warps)
        const int ew = warp & 3;                 // TMEM lane quarter this warp may read
        const int cg = warp >> 2;                // column group of the tile this warp scans
        const int row = ew * 32 + lane;          // query row inside the tile
        uint32_t tile_n = 0;
        SegIter it(p.n_qtiles, p.n_ttiles, p.units_per_cta, blockIdx.x);
        int qtile, t_begin, t_end, seg;
        while (it.next(qtile, t_begin, t_end, seg)) {
            float bs[TOPK];
            int bi[TOPK];
#pragma unroll
            for (int j = 0; j < TOPK; j++) { bs[j] = INFINITY; bi[j] = -1; }
            const int qrow = qtile * BM + row;
            const float slack = slack_of(qrow < p.nq ? p.qn[qrow] : 0.f, __uint_as_float(*p.tn_max_bits), (float)KAPPA);
            for (int tt = t_begin; tt < t_end; tt++, tile_n++) {
                const uint32_t acc = tile_n & 1;
                mbar_wait(&nfull[acc], (tile_n >> 1) & 1);
                mbar_wait(&pipe.tfull[acc], (tile_n >> 1) & 1);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + acc * BN + cg * EPI_COLS;
                // |t|^2 of this warp's columns: every lane reads the same 16 bytes (shared-memory broadcast)
                const float4* tn4 = reinterpret_cast<const float4*>(tn_smem + acc * BN + cg * EPI_COLS);
                const int colbase = tt * BN + cg * EPI_COLS;
                // TMEM -> registers double buffered: the load of chunk c+1 flies while chunk c is scanned
                uint32_t va[32], vb[32];
                tc_ld32(taddr, va);
#pragma unroll 1
                for (int cc = 0; cc < EPI_COLS / 32; cc += 2) {
                    tc_wait_ld32(va);
                    tc_ld32(taddr + (cc + 1) * 32, vb);
                    scan_chunk(va, taddr + cc * 32, tn4 + cc * 8, colbase + cc * 32, slack, bs, bi);
                    tc_wait_ld32(vb);
                    if (cc + 2 < EPI_COLS / 32) tc_ld32(taddr + (cc + 2) * 32, va);
                    scan_chunk(vb, taddr + (cc + 1) * 32, tn4 + (cc + 1) * 8, colbase + (cc + 1) * 32, slack, bs, bi);
                }
                // accumulator drained: hand it back to the MMA warp
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&pipe.tempty[acc]);
            }
            const int qg = qtile * BM + row;
            if (qg < p.nq) {
                const size_t o = ((size_t)qg * p.n_seg + seg) * EPI_GROUPS + cg;
                *reinterpret_cast<int4*>(p.cand_idx + o * TOPK) = make_int4(bi[0], bi[1], bi[2], bi[3]);
                *reinterpret_cast<float4*>(p.cand_s + o * TOPK) = make_float4(bs[0], bs[1], bs[2], bs[3]);
                p.cand_thr[o] = fminf(bs[3], __fadd_rn(bs[1], slack));
            }
        }
    }

    tmem_free(warp == W_ALLOC, tmem_base);
}

// ------------------------------------------------------------------------------------------
// refine: exact distances of the candidates, top-2, certificate
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool lex_less(double d, int i, double bd, int bi) { return d < bd || (d == bd && i < bi); }

// one warp per query; lane j owns candidates j, j + 32, ... (n_groups * TOPK <= 32 * SPL, n_groups = segments x column groups;
// SPL = 2 for up to four segments per query row, 4 when a short query set is cut finer to fill the machine)
template <int SPL>
__global__ void __launch_bounds__(256)
refine_kernel(const float* __restrict__ q, int nq, const float* __restrict__ t, int nt, int dim, int n_groups, int topk, double kappa,
              double f16_abs, const int32_t* __restrict__ cand_idx, const float* __restrict__ cand_s, const float* __restrict__ cand_thr,
              unsigned* __restrict__ misc /* [0] re-scan count, [1] max |t|^2 bits, [2] max deviation bits, [5], [6]: below */,
              int32_t* __restrict__ idx2, float* __restrict__ dist2, double* __restrict__ d2out,
              int32_t* __restrict__ rescan_list)
{
    const int qi = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (qi >= nq) return;
    const int ncand = n_groups * topk;
    const float* qr = q + (size_t)qi * dim;

    // certificate inputs first: the smallest per-list bound (every non-candidate of a list has an approximate
    // score >= its bound; lists that were never written keep the 0x7f.. fill = "no non-candidates")
    float thr = INFINITY;
    for (int l = lane; l < n_groups; l += 32) {
        float b = cand_thr[(size_t)qi * n_groups + l];
        thr = fminf(thr, b > 3.0e38f ? INFINITY : b);
    }
    for (int o = 16; o > 0; o >>= 1) thr = fminf(thr, __shfl_xor_sync(0xffffffffu, thr, o));

    // exact distances of the candidates that matter: a listed column whose approximate score is not below that bound
    // is covered by the certificate like any unlisted column, so its exact distance is not needed.  The ones that are left
    // (usually two to six of the 64 slots) are compacted through shared memory so that one pass of the warp evaluates
    // them, and the query row is converted to fp64 ONCE per warp (the fp32 -> fp64 conversions, not the FMAs, were the
    // limiter: 128 per candidate).  Each candidate still gets the oracle's fma chain in the oracle's order.
    __shared__ double q_sh[8][128];
    __shared__ int c_idx[8][32 * SPL];
    __shared__ float c_sc[8][32 * SPL];
    const int wq = threadIdx.x >> 5;
    for (int k = lane; k < dim; k += 32) q_sh[wq][k] = (double)qr[k];
    int n_act;
    {
        const unsigned lt = (1u << lane) - 1u;
        n_act = 0;
#pragma unroll
        for (int s = 0; s < SPL; s++) {
            const int c = lane + 32 * s;
            const int ti = c < ncand ? cand_idx[(size_t)qi * ncand + c] : -1;
            const float s2 = (c < ncand && ti >= 0) ? cand_s[(size_t)qi * ncand + c] : INFINITY;   // unused list slots are -1 / unset
            const bool act = ti >= 0 && ti < nt && (s2 < thr || !(thr < INFINITY));
            const unsigned mk = __ballot_sync(0xffffffffu, act);
            if (act) { const int pos = n_act + __popc(mk & lt); c_idx[wq][pos] = ti; c_sc[wq][pos] = s2; }
            n_act += __popc(mk);
        }
    }
    __syncwarp();
    double d[SPL];
    int id[SPL];
    float sc[SPL];
#pragma unroll
    for (int s = 0; s < SPL; s++) {
        const int c = lane + 32 * s;
        d[s] = INFINITY; id[s] = 0x7fffffff; sc[s] = INFINITY;
        if (32 * s < n_act) {                                  // warp-uniform: the second pass rarely runs
            if (c < n_act) {
                const int ti = c_idx[wq][c];
                sc[s] = c_sc[wq][c];
                const float* tr = t + (size_t)ti * dim;
                double a = 0.0;
                // 16 floats of the train row in flight at a time (the loads, not the chain, set the pace otherwise: one
                // L2 round trip per 4 terms); the chain itself stays in index order
                int k = 0;
                for (; k + 16 <= dim; k += 16) {
                    float4 y[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) y[u] = *reinterpret_cast<const float4*>(tr + k + 4 * u);
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        double e;
                        e = __dsub_rn(q_sh[wq][k + 4 * u], (double)y[u].x); a = __fma_rn(e, e, a);
                        e = __dsub_rn(q_sh[wq][k + 4 * u + 1], (double)y[u].y); a = __fma_rn(e, e, a);
                        e = __dsub_rn(q_sh[wq][k + 4 * u + 2], (double)y[u].z); a = __fma_rn(e, e, a);
                        e = __dsub_rn(q_sh[wq][k + 4 * u + 3], (double)y[u].w); a = __fma_rn(e, e, a);
                    }
                }
                for (; k < dim; k += 4) {
                    float4 y = *reinterpret_cast<const float4*>(tr + k);
                    double e;
                    e = __dsub_rn(q_sh[wq][k], (double)y.x); a = __fma_rn(e, e, a);
                    e = __dsub_rn(q_sh[wq][k + 1], (double)y.y); a = __fma_rn(e, e, a);
                    e = __dsub_rn(q_sh[wq][k + 2], (double)y.z); a = __fma_rn(e, e, a);
                    e = __dsub_rn(q_sh[wq][k + 3], (double)y.w); a = __fma_rn(e, e, a);
                }
                d[s] = a; id[s] = ti;
            }
        }
    }
    double qn = 0.0;
    for (int k = lane; k < dim; k += 32) { double x = q_sh[wq][k]; qn += x * x; }
    for (int o = 16; o > 0; o >>= 1) qn += __shfl_xor_sync(0xffffffffu, qn, o);
    const double tn_max = (double)__uint_as_float(misc[1]);
    const double scale = qn + tn_max;
    // observed |approximate - exact| over the candidates, in units of (|q|^2 + max|t|^2)
    float dev = 0.f;
#pragma unroll
    for (int s = 0; s < SPL; s++)
        if (id[s] != 0x7fffffff && scale > 0.0) dev = fmaxf(dev, (float)(fabs((double)sc[s] + qn - d[s]) / scale));
    for (int o = 16; o > 0; o >>= 1) dev = fmaxf(dev, __shfl_xor_sync(0xffffffffu, dev, o));

    // lane-local order (the two smallest of the lane's entries to slots 0 and 1), then two warp-wide lexicographic minima
#pragma unroll
    for (int s = 1; s < SPL; s++) {
        if (lex_less(d[s], id[s], d[1], id[1])) { double x = d[1]; d[1] = d[s]; d[s] = x; int y = id[1]; id[1] = id[s]; id[s] = y; }
        if (lex_less(d[1], id[1], d[0], id[0])) { double x = d[0]; d[0] = d[1]; d[1] = x; int y = id[0]; id[0] = id[1]; id[1] = y; }
    }
    double B0 = d[0]; int I0 = id[0];
    for (int o = 16; o > 0; o >>= 1) {
        double od = __shfl_xor_sync(0xffffffffu, B0, o); int oi = __shfl_xor_sync(0xffffffffu, I0, o);
        if (lex_less(od, oi, B0, I0)) { B0 = od; I0 = oi; }
    }
    // the lane holding the winner promotes its second entry (candidate indices are distinct)
    double m = d[0]; int mi = id[0];
    if (mi == I0) { m = d[1]; mi = id[1]; }
    double B1 = m; int I1 = mi;
    for (int o = 16; o > 0; o >>= 1) {
        double od = __shfl_xor_sync(0xffffffffu, B1, o); int oi = __shfl_xor_sync(0xffffffffu, I1, o);
        if (lex_less(od, oi, B1, I1)) { B1 = od; I1 = oi; }
    }

    if (lane == 0) {
        // (same-address atomics from every warp were the whole cost of this kernel: 135 us for 100k queries)
        if (dev > 0.f && __float_as_uint(dev) > *reinterpret_cast<volatile unsigned*>(misc + 2)) atomicMax(misc + 2, __float_as_uint(dev));
        const double eps = kappa * scale;
        // non-finite input anywhere (NaN compares false, inf norms) -> exact re-scan
        bool finite_in = scale < (double)INFINITY && scale == scale;
        // f16 operands (f16_abs >= 0, knn_tc1.cu): the call's range guard (misc[5]) and the absolute error of subnormal operands;
        // queries that fail either go to the re-scan and are counted in misc[6]
        bool in_range = true;
        if (f16_abs >= 0.0 && finite_in) {
            const double sub = 0x1p-24 * sqrt((double)dim) * (2.0 * sqrt(qn) + sqrt(tn_max)) + 0x1p-36;
            in_range = misc[5] == 0u && sub <= f16_abs * scale;
            if (!in_range) atomicAdd(misc + 6, 1u);
        }
        bool certified = finite_in && in_range && I1 != 0x7fffffff &&
                         (!(thr < INFINITY) /* every train row was a candidate */ || B1 < (double)thr + qn - eps);
        if (certified) {
            if (idx2) { idx2[2 * qi] = I0; idx2[2 * qi + 1] = I1; }
            if (dist2) { dist2[2 * qi] = (float)sqrt(B0); dist2[2 * qi + 1] = (float)sqrt(B1); }
            if (d2out) { d2out[2 * qi] = B0; d2out[2 * qi + 1] = B1; }
        } else {
            int pos = (int)atomicAdd(misc, 1u);
            rescan_list[pos] = qi;
        }
    }
}

// topk must be a power of two, n_lists * topk <= 128
// misc words of a tcgen05 call: [0] re-scan count of THIS call (also the length of its re-scan list), [1] max |t|^2 bits,
// [2] max deviation bits, [3] max |q|^2 bits, [4] re-scan count summed over the query chunks of one host call,
// [5] f16 range guard raised (by the prep of any chunk), [6] queries the f16 range checks sent to the re-scan (all chunks)
__global__ void misc_reset_kernel(int32_t* misc) { misc[0] = 0; misc[3] = 0; }
__global__ void misc_accum_kernel(int32_t* misc) { misc[4] += misc[0]; }
int tc_misc_begin(erp_ctx* ctx, int32_t* misc)
{
    if (ctx->tc_chunk == 0) {
        ERP_CUDA(cudaMemsetAsync(misc, 0, 8 * sizeof(int32_t), ctx->stream));
    } else {
        misc_reset_kernel<<<1, 1, 0, ctx->stream>>>(misc);
        ERP_LAUNCH(ctx, "misc_reset_kernel");
    }
    return ERP_OK;
}
int tc_misc_end(erp_ctx* ctx, int32_t* misc)
{
    misc_accum_kernel<<<1, 1, 0, ctx->stream>>>(misc);
    ERP_LAUNCH(ctx, "misc_accum_kernel");
    return ERP_OK;
}

int refine_launch(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim, int n_lists, int topk, double kappa,
                  double f16_abs, const int32_t* cand, const float* cand_s, const float* cand_thr, unsigned* misc, int32_t* d_idx2, float* d_dist2,
                  double* d_d2, int32_t* rescan_list)
{
    if (n_lists * topk > 128) { set_error("refine: %d candidate slots per query", n_lists * topk); return ERP_E_LIMIT; }
    if (n_lists * topk <= 64)
        refine_kernel<2><<<cdiv(nq, 8), 256, 0, ctx->stream>>>(d_q, nq, d_t, nt, dim, n_lists, topk, kappa, f16_abs, cand, cand_s, cand_thr, misc,
                                                               d_idx2, d_dist2, d_d2, rescan_list);
    else
        refine_kernel<4><<<cdiv(nq, 8), 256, 0, ctx->stream>>>(d_q, nq, d_t, nt, dim, n_lists, topk, kappa, f16_abs, cand, cand_s, cand_thr, misc,
                                                               d_idx2, d_dist2, d_d2, rescan_list);
    ERP_LAUNCH(ctx, "refine_kernel");
    return ERP_OK;
}

bool knn2_tc_supported(int nq, int nt, int dim) { return nq >= 1 && nt >= 2 && dim >= 4 && dim % 4 == 0 && dim <= 128; }

// AUTO policy: tensor cores once the problem is large enough to amortise the extra passes, and then the one-product
// engine (knn_tc1.cu), measured faster than 3xTF32 at every size where a tensor engine pays at all
// (20k x 20k x 64: 0.14 vs 0.27 ms, 50k x 50k: 0.54 vs 1.20 ms, 100k x 100k: 1.7 vs 4.2 ms)
bool knn2_tc_preferred(int nq, int nt, int dim)
{
    return knn2_tc_supported(nq, nt, dim) && (double)nq * (double)nt >= 4.0e6;
}

int knn2_exact_rescan(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                      const int32_t* d_list, const int32_t* d_count, int max_rows,
                      int32_t* d_idx2, float* d_dist2, double* d_d2);

int knn2_tc(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
            int32_t* d_idx2, float* d_dist2, double* d_d2)
{
    if (!knn2_tc_supported(nq, nt, dim)) { set_error("tcgen05 engine: unsupported shape nq=%d nt=%d dim=%d", nq, nt, dim); return ERP_E_DIM; }
    const int kch = (dim + KC - 1) / KC, dpad = kch * KC;
    const int n_qtiles = cdiv(nq, BM), n_ttiles = cdiv(nt, BN);
    const StreamK plan = stream_k_plan(n_qtiles, n_ttiles, ctx->sm_count, MAX_SEG);
    const int n_seg = plan.n_seg, n_lists = n_seg * EPI_GROUPS;

    int st = ERP_OK;
    float* qs = ctx->scratch<float>(S_TC_Q, (size_t)nq * 2 * dpad, &st);
    float* ts = ctx->scratch<float>(S_TC_T, (size_t)nt * 2 * dpad, &st);
    float* tn = ctx->scratch<float>(S_TC_TN, (size_t)n_ttiles * BN, &st);
    int32_t* cand = ctx->scratch<int32_t>(S_TC_CAND, (size_t)nq * n_lists * (TOPK * 2 + 1), &st);
    float* qn = ctx->scratch<float>(S_TC_QN, (size_t)nq + 8, &st);
    int32_t* list = ctx->scratch<int32_t>(S_TC_LIST, (size_t)nq + 8, &st);
    int32_t* misc = ctx->scratch<int32_t>(S_TC_MISC, 8, &st);     // [0] re-scan count, [1] max |t|^2 bits, [2] max deviation bits
    ERP_TRY(st);
    float* cand_s = reinterpret_cast<float*>(cand + (size_t)nq * n_lists * TOPK);
    float* cand_thr = cand_s + (size_t)nq * n_lists * TOPK;
    ERP_CUDA(cudaMemsetAsync(cand_thr, 0x7f, (size_t)nq * n_lists * sizeof(float), ctx->stream));              // ~3.4e38: "unbounded"
    ERP_TRY(tc_misc_begin(ctx, misc));
    ERP_CUDA(cudaMemsetAsync(cand, 0xFF, (size_t)nq * n_lists * TOPK * sizeof(int32_t), ctx->stream));   // index -1: empty slot

    ERP_TRY(launch_prep(ctx, d_q, nq, dim, dpad, -2.0f, qs, qn, nq, reinterpret_cast<unsigned*>(misc + 3)));
    if (ctx->tc_chunk == 0) ERP_TRY(launch_prep(ctx, d_t, nt, dim, dpad, 1.0f, ts, tn, n_ttiles * BN, reinterpret_cast<unsigned*>(misc + 1)));

    CUtensorMap mq, mt;
    ERP_TRY(make_map(&mq, qs, nq, 2 * dpad, BM, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4));
    ERP_TRY(make_map(&mt, ts, nt, 2 * dpad, BN, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4));
    TcParams p;
    p.nq = nq; p.nt = nt; p.n_qtiles = n_qtiles; p.n_ttiles = n_ttiles; p.units_per_cta = plan.units_per_cta; p.n_seg = n_seg;
    p.tn = tn; p.cand_idx = cand; p.cand_s = cand_s; p.cand_thr = cand_thr; p.qn = qn;
    p.tn_max_bits = reinterpret_cast<const unsigned*>(misc + 1);

    if (ctx->tc_chunk == 0) ERP_CUDA(record_timing(ctx, ctx->ev_k0));
    switch (kch) {
    case 1: ERP_TRY(launch_tc_kernel<knn2_tc_kernel<1>>(ctx, "knn2_tc_kernel", plan.grid, TC_THREADS, tc_smem(1), mq, mt, p)); break;
    case 2: ERP_TRY(launch_tc_kernel<knn2_tc_kernel<2>>(ctx, "knn2_tc_kernel", plan.grid, TC_THREADS, tc_smem(2), mq, mt, p)); break;
    case 3: ERP_TRY(launch_tc_kernel<knn2_tc_kernel<3>>(ctx, "knn2_tc_kernel", plan.grid, TC_THREADS, tc_smem(3), mq, mt, p)); break;
    default: ERP_TRY(launch_tc_kernel<knn2_tc_kernel<4>>(ctx, "knn2_tc_kernel", plan.grid, TC_THREADS, tc_smem(4), mq, mt, p)); break;
    }
    ERP_CUDA(record_timing(ctx, ctx->ev_k1));

    ERP_TRY(refine_launch(ctx, d_q, nq, d_t, nt, dim, n_lists, TOPK, KAPPA, -1.0, cand, cand_s, cand_thr, reinterpret_cast<unsigned*>(misc),
                          d_idx2, d_dist2, d_d2, list));
    ERP_TRY(knn2_exact_rescan(ctx, d_q, nq, d_t, nt, dim, list, misc, nq, d_idx2, d_dist2, d_d2));
    ERP_TRY(tc_misc_end(ctx, misc));

    set_knn_stats(ctx, ERP_ENGINE_TCGEN05, false, n_seg, plan.units_per_cta, plan.grid, misc);
    return ERP_OK;
}

} // namespace erp
