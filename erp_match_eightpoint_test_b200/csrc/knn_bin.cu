// knn_bin.cu -- exact Hamming 2-NN of binary descriptors (ORB, AKAZE/MLDB, BRISK, FREAK, LATCH: 1..64 bytes per row).
//
// sm_100 has no 1-bit tensor product.  Every bit is expanded to an int8 of +1 (set) or -1 (clear), so for two n-bit rows
//     dot = n - 2 * Hamming
// and one tcgen05.mma.kind::i8 GEMM (s8 x s8 -> s32) yields the EXACT distance in its accumulator: no norm step, no
// rounding certificate, no refine or re-scan pass.  A kind::i8 instruction (K = 32) reads the same 32 bytes per operand
// row as a kind::f16 K = 16 step, so the tile shape and the query-pair pipeline of knn_tc1.cu (tc_common.cuh: PairPipe)
// carry over.  K padding is 0 on both sides and contributes nothing.
//
// Ties are the normal case for Hamming distances (a third of the queries of random 256-bit rows tie at the second
// position), so every list is kept exactly in (H, trainIdx) order: the lowest index wins a tie everywhere.
#include "tc_common.cuh"

#include <climits>

namespace erp {

constexpr int B_BM = 128;                 // queries per sub-tile (UMMA M)
constexpr int B_BN = 256;                 // train rows per tile (UMMA N)
constexpr int B_QCH = B_BM * 128;         // 16 KB: one 128-byte k chunk of a query sub-tile
constexpr int B_TCH = B_BN * 128;         // 32 KB: one 128-byte k chunk of a train tile
constexpr int B_EPI_GROUPS = 2;
constexpr int B_EPI_THREADS = B_EPI_GROUPS * 128;
constexpr int B_THREADS = 128 + B_EPI_THREADS;
constexpr int B_EPI_COLS = B_BN / B_EPI_GROUPS;
constexpr int B_MAX_SEG = 16;
constexpr int B_BARS = 256;
// instruction descriptor (PTX ISA, tcgen05 instruction descriptor for .kind::i8): D format s32 (2) in bits [4,6),
// A and B format signed 8-bit (1) in bits [7,10) and [10,13), both K-major, N >> 3 in bits [17,23), M >> 4 in [24,29)
constexpr uint32_t B_IDESC_I8 = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(B_BN >> 3) << 17) | ((uint32_t)(B_BM >> 4) << 24);

// two resident query sub-tiles share every train tile while shared memory leaves a look-ahead chunk (KCH <= 3)
__host__ __device__ constexpr int b_sub(int kch) { return kch <= 3 ? 2 : 1; }
__host__ __device__ constexpr int b_slots(int kch) { return (TC_SMEM_LIMIT - b_sub(kch) * kch * B_QCH - B_BARS) / B_TCH; }
__host__ __device__ constexpr int b_smem(int kch) { return b_sub(kch) * kch * B_QCH + b_slots(kch) * B_TCH + B_BARS; }

// ---- operands: packed bits -> int8 rows of +-1, K padding 0 (bit i of byte k is element 8k + i on both sides)
struct BinJob { const uint8_t* x; int n; int8_t* out; int blocks; };

__global__ void __launch_bounds__(256)
bin_prep_kernel(const BinJob a, const BinJob b, int nbytes, int kpad)
{
    const bool second = (int)blockIdx.x >= a.blocks;
    const BinJob& j = second ? b : a;
    const int per_row = kpad / 8;                                // output bytes come in groups of 8 (one input byte)
    const long i = (long)((int)blockIdx.x - (second ? a.blocks : 0)) * 256 + threadIdx.x;
    if (i >= (long)j.n * per_row) return;
    const int row = (int)(i / per_row), k = (int)(i % per_row);
    uint2 o = make_uint2(0u, 0u);
    if (k < nbytes) {
        const uint32_t v = j.x[(size_t)row * nbytes + k];
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int bit = 0; bit < 4; bit++) {
            lo |= ((v >> bit) & 1u ? 0x01u : 0xFFu) << (8 * bit);
            hi |= ((v >> (bit + 4)) & 1u ? 0x01u : 0xFFu) << (8 * bit);
        }
        o = make_uint2(lo, hi);
    }
    *reinterpret_cast<uint2*>(j.out + (size_t)row * kpad + 8 * k) = o;
}

struct BinParams {
    int nq, nt, nbits;
    int n_qpairs, n_ttiles;
    int units_per_cta;
    int n_seg;                    // lists per query = n_seg x B_EPI_GROUPS, 2 keys each
    unsigned long long* cand;     // (H << 32 | trainIdx), ascending = (distance, index) order; ~0 = empty
};

// best column of 32 accumulator values as (acc << 7 | 127 - column): the maximum is the largest dot product (smallest
// distance), and among equal ones the lowest column.  CHECK: skip columns >= lim (past the last train row) and excl.
template <bool CHECK>
__device__ __forceinline__ int best_of32(const uint32_t (&v)[32], int c0, int lim, int excl, int m)
{
#pragma unroll
    for (int j = 0; j < 32; j++) {
        const int c = c0 + j;
        int k = (int)v[j] * 128 + (127 - c);
        if (CHECK && (c >= lim || c == excl)) k = INT_MIN;
        m = max(m, k);
    }
    return m;
}

template <int KCH>
__global__ void __launch_bounds__(B_THREADS, 1)
knn2_bin_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_t, const BinParams p)
{
    constexpr int NS = b_slots(KCH), SUB = b_sub(KCH);
    static_assert(NS >= KCH + 1, "T ring must hold one tile plus a chunk of look-ahead");
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint8_t* q_smem = smem;                                   // [SUB][KCH] chunks
    uint8_t* t_smem = smem + SUB * KCH * B_QCH;               // NS slots
    uint64_t* bars = reinterpret_cast<uint64_t*>(t_smem + NS * B_TCH);
    using Pipe = PairPipe<SUB, KCH, NS, B_BM, B_BN, 128>;
    const Pipe pipe(q_smem, t_smem, bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + Pipe::N_BARS);
    static_assert(Pipe::N_BARS * 8 + 4 <= B_BARS, "barrier block");
    static_assert(b_smem(KCH) <= TC_SMEM_LIMIT, "shared memory budget");

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int W_ALLOC = B_EPI_THREADS / 32, W_TMA = W_ALLOC + 2, W_MMA = W_ALLOC + 3;   // W_ALLOC + 1 idles

    if (warp == W_TMA && lane == 0) { tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_t); }
    if (warp == W_MMA && lane == 0) pipe.init(B_EPI_THREADS / 32);
    const uint32_t tmem_base = tmem_alloc(warp == W_ALLOC, tmem_slot);

    // the feeder warpgroup needs few registers; the eight epilogue warps take them over (128 accumulator columns in flight)
    if (warp >= W_ALLOC) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
    if (warp == W_TMA) {
        // ================================================================ TMA producer
        if (lane == 0) pipe.produce(&map_q, &map_t, SegIter(p.n_qpairs, p.n_ttiles, p.units_per_cta, blockIdx.x));
    } else if (warp == W_MMA) {
        // ================================================================ MMA issuer
        if (lane == 0)
            pipe.issue(tmem_base, SegIter(p.n_qpairs, p.n_ttiles, p.units_per_cta, blockIdx.x),
                       [](uint32_t d_tmem, uint32_t q, int c, uint32_t b) { mma_chunk<tc_mma_i8>(d_tmem, q + c * B_QCH, b, B_IDESC_I8, c != 0); },
                       [](int, uint32_t, uint32_t) {});
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
            unsigned long long b0[SUB], b1[SUB];
#pragma unroll
            for (int sub = 0; sub < SUB; sub++) b0[sub] = b1[sub] = ~0ull;
            for (int tt = t0; tt < t1; tt++) {
                const int colbase = tt * B_BN + cg * B_EPI_COLS;
                const int lim = p.nt - colbase;          // columns >= lim are zero padding rows (they would score nbits / 2)
#pragma unroll
                for (int sub = 0; sub < SUB; sub++, tile_n++) {
                    const uint32_t acc = tile_n & 1;
                    mbar_wait(&pipe.tfull[acc], (tile_n >> 1) & 1);
                    tc_fence_after();
                    const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + acc * B_BN + cg * B_EPI_COLS;
                    uint32_t va[32], vb[32], vc[32], vd[32];
                    pipe.drain(taddr, acc, va, vb, vc, vd);
                    int m;
                    if (lim >= B_EPI_COLS) {
                        m = best_of32<false>(va, 0, 0, -1, INT_MIN);
                        m = best_of32<false>(vb, 32, 0, -1, m);
                        m = best_of32<false>(vc, 64, 0, -1, m);
                        m = best_of32<false>(vd, 96, 0, -1, m);
                    } else {
                        m = best_of32<true>(va, 0, lim, -1, INT_MIN);
                        m = best_of32<true>(vb, 32, lim, -1, m);
                        m = best_of32<true>(vc, 64, lim, -1, m);
                        m = best_of32<true>(vd, 96, lim, -1, m);
                    }
                    // insert while the tile's best beats the runner-up; after two inserts from one tile every other column
                    // of it ranks behind both, so at most two rounds
#pragma unroll 1
                    for (int round = 0; round < 2 && m != INT_MIN; round++) {
                        const int col = 127 - (m & 127);
                        const unsigned h = (unsigned)(p.nbits - (m >> 7)) >> 1;
                        const unsigned long long key = ((unsigned long long)h << 32) | (unsigned)(colbase + col);
                        if (!(key < b1[sub])) break;
                        if (key < b0[sub]) { b1[sub] = b0[sub]; b0[sub] = key; }
                        else b1[sub] = key;
                        if (round == 1) break;
                        m = best_of32<true>(va, 0, lim, col, INT_MIN);
                        m = best_of32<true>(vb, 32, lim, col, m);
                        m = best_of32<true>(vc, 64, lim, col, m);
                        m = best_of32<true>(vd, 96, lim, col, m);
                    }
                }
            }
#pragma unroll
            for (int sub = 0; sub < SUB; sub++) {
                const int qg = (qp * SUB + sub) * B_BM + row;
                if (qg < p.nq) {
                    const size_t l = ((size_t)qg * p.n_seg + seg) * B_EPI_GROUPS + cg;
                    *reinterpret_cast<ulonglong2*>(p.cand + 2 * l) = make_ulonglong2(b0[sub], b1[sub]);
                }
            }
        }
    }

    tmem_free(warp == W_ALLOC, tmem_base);
}

// the n_lists x 2 keys of a query -> its two nearest in (distance, index) order
__global__ void bin_merge_kernel(const unsigned long long* __restrict__ cand, int nq, int n_keys,
                                 int32_t* __restrict__ idx2, float* __restrict__ dist2, double* __restrict__ d2)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    unsigned long long k0 = ~0ull, k1 = ~0ull;
    const unsigned long long* c = cand + (size_t)q * n_keys;
    for (int i = 0; i < n_keys; i++) {
        const unsigned long long k = c[i];
        if (k < k0) { k1 = k0; k0 = k; }
        else if (k < k1) k1 = k;
    }
    const unsigned long long k[2] = {k0, k1};
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const bool ok = k[j] != ~0ull;
        const float h = ok ? (float)(unsigned)(k[j] >> 32) : INFINITY;
        if (idx2) idx2[2 * q + j] = ok ? (int32_t)(uint32_t)k[j] : -1;
        if (dist2) dist2[2 * q + j] = h;
        if (d2) d2[2 * q + j] = (double)h;
    }
}

// ---- SIMT engine: __popc on 32-bit words, one query per thread, train rows staged through shared memory.
// W: words per row rounded up to a power of two (the zero words of both sides XOR to nothing).
constexpr int BX_THREADS = 128;

__device__ __forceinline__ void load_words(const uint8_t* __restrict__ r, int nbytes, uint32_t* w, int W)
{
    for (int i = 0; i < W; i++) {
        uint32_t v = 0;
        for (int b = 0; b < 4; b++) {
            const int k = 4 * i + b;
            if (k < nbytes) v |= (uint32_t)r[k] << (8 * b);
        }
        w[i] = v;
    }
}

template <int W>
__global__ void __launch_bounds__(BX_THREADS)
knn2_bin_exact_kernel(const uint8_t* __restrict__ q, int nq, const uint8_t* __restrict__ t, int nt, int nbytes,
                      int32_t* __restrict__ idx2, float* __restrict__ dist2, double* __restrict__ d2)
{
    __shared__ uint32_t ts[BX_THREADS][W];
    const int qi = blockIdx.x * BX_THREADS + threadIdx.x;
    uint32_t qw[W];
    if (qi < nq) load_words(q + (size_t)qi * nbytes, nbytes, qw, W);
    else for (int i = 0; i < W; i++) qw[i] = 0;
    int d0 = INT_MAX, d1 = INT_MAX, i0 = -1, i1 = -1;
    for (int t0 = 0; t0 < nt; t0 += BX_THREADS) {
        __syncthreads();
        if (t0 + (int)threadIdx.x < nt) load_words(t + (size_t)(t0 + threadIdx.x) * nbytes, nbytes, ts[threadIdx.x], W);
        __syncthreads();
        const int n = nt - t0 < BX_THREADS ? nt - t0 : BX_THREADS;
        for (int j = 0; j < n; j++) {
            int d = 0;
#pragma unroll
            for (int i = 0; i < W; i++) d += __popc(qw[i] ^ ts[j][i]);
            // ascending train index and strict <: a tie keeps the lower index
            if (d < d1) {
                if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = t0 + j; }
                else { d1 = d; i1 = t0 + j; }
            }
        }
    }
    if (qi >= nq) return;
    const int di[2] = {d0, d1}, ii[2] = {i0, i1};
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const float h = ii[j] >= 0 ? (float)di[j] : INFINITY;
        if (idx2) idx2[2 * qi + j] = ii[j];
        if (dist2) dist2[2 * qi + j] = h;
        if (d2) d2[2 * qi + j] = (double)h;
    }
}

// The kind::i8 engine is already 2.5x faster than SIMT at 1000 x 1000 x 32 B (DESIGN.md 4.8: 0.042 vs 0.103 ms per call,
// B200); below 1e6 pairs, where nothing was measured, SIMT's single launch is kept.
bool knn2_bin_preferred(int nq, int nt) { return (double)nq * (double)nt >= 1.0e6; }

int knn2_bin(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes, bool tc,
             int32_t* d_idx2, float* d_dist2, double* d_d2)
{
    if (!tc) {
        set_knn_stats(ctx, ERP_ENGINE_EXACT_SIMT, true, 1, cdiv(nq, BX_THREADS), 0, nullptr);
        const int W = nbytes <= 8 ? 2 : nbytes <= 16 ? 4 : nbytes <= 32 ? 8 : 16;
        const int grid = cdiv(nq, BX_THREADS);
        if (ctx->tc_chunk == 0) ERP_CUDA(record_timing(ctx, ctx->ev_k0));
        switch (W) {
        case 2: knn2_bin_exact_kernel<2><<<grid, BX_THREADS, 0, ctx->stream>>>(d_q, nq, d_t, nt, nbytes, d_idx2, d_dist2, d_d2); break;
        case 4: knn2_bin_exact_kernel<4><<<grid, BX_THREADS, 0, ctx->stream>>>(d_q, nq, d_t, nt, nbytes, d_idx2, d_dist2, d_d2); break;
        case 8: knn2_bin_exact_kernel<8><<<grid, BX_THREADS, 0, ctx->stream>>>(d_q, nq, d_t, nt, nbytes, d_idx2, d_dist2, d_d2); break;
        default: knn2_bin_exact_kernel<16><<<grid, BX_THREADS, 0, ctx->stream>>>(d_q, nq, d_t, nt, nbytes, d_idx2, d_dist2, d_d2); break;
        }
        ERP_LAUNCH(ctx, "knn2_bin_exact_kernel");
        ERP_CUDA(record_timing(ctx, ctx->ev_k1));
        return ERP_OK;
    }
    const int kch = (nbytes + 15) / 16, kpad = kch * 128;
    const int n_qpairs = cdiv(nq, B_BM * b_sub(kch)), n_ttiles = cdiv(nt, B_BN);
    const StreamK plan = stream_k_plan(n_qpairs, n_ttiles, ctx->sm_count, B_MAX_SEG);
    const int n_seg = plan.n_seg;
    const int n_keys = n_seg * B_EPI_GROUPS * 2;

    int st = ERP_OK;
    int8_t* qs = ctx->scratch<int8_t>(S_TC_Q, (size_t)nq * kpad, &st);
    int8_t* ts = ctx->scratch<int8_t>(S_TC_T, (size_t)nt * kpad, &st);
    unsigned long long* cand = ctx->scratch<unsigned long long>(S_TC_CAND, (size_t)nq * n_keys, &st);
    ERP_TRY(st);
    // lists of segments a query pair does not have stay empty
    ERP_CUDA(cudaMemsetAsync(cand, 0xFF, (size_t)nq * n_keys * sizeof(unsigned long long), ctx->stream));
    // a later query chunk of one host call finds the train operand prepared by the first
    BinJob jq = {d_q, nq, qs, 0};
    BinJob jt = {ctx->tc_chunk == 0 ? d_t : nullptr, nt, ts, 0};
    jq.blocks = (int)(((long)nq * (kpad / 8) + 255) / 256);
    jt.blocks = jt.x ? (int)(((long)nt * (kpad / 8) + 255) / 256) : 0;
    bin_prep_kernel<<<jq.blocks + jt.blocks, 256, 0, ctx->stream>>>(jq, jt, nbytes, kpad);
    ERP_LAUNCH(ctx, "bin_prep_kernel");

    CUtensorMap mq, mt;
    ERP_TRY(make_map(&mq, qs, nq, kpad, B_BM, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1));
    ERP_TRY(make_map(&mt, ts, nt, kpad, B_BN, CU_TENSOR_MAP_DATA_TYPE_UINT8, 1));
    BinParams p;
    p.nq = nq; p.nt = nt; p.nbits = 8 * nbytes; p.n_qpairs = n_qpairs; p.n_ttiles = n_ttiles; p.units_per_cta = plan.units_per_cta;
    p.n_seg = n_seg; p.cand = cand;

    if (ctx->tc_chunk == 0) ERP_CUDA(record_timing(ctx, ctx->ev_k0));
    switch (kch) {
    case 1: ERP_TRY(launch_tc_kernel<knn2_bin_kernel<1>>(ctx, "knn2_bin_kernel", plan.grid, B_THREADS, b_smem(1), mq, mt, p)); break;
    case 2: ERP_TRY(launch_tc_kernel<knn2_bin_kernel<2>>(ctx, "knn2_bin_kernel", plan.grid, B_THREADS, b_smem(2), mq, mt, p)); break;
    case 3: ERP_TRY(launch_tc_kernel<knn2_bin_kernel<3>>(ctx, "knn2_bin_kernel", plan.grid, B_THREADS, b_smem(3), mq, mt, p)); break;
    default: ERP_TRY(launch_tc_kernel<knn2_bin_kernel<4>>(ctx, "knn2_bin_kernel", plan.grid, B_THREADS, b_smem(4), mq, mt, p)); break;
    }
    ERP_CUDA(record_timing(ctx, ctx->ev_k1));
    bin_merge_kernel<<<cdiv(nq, 256), 256, 0, ctx->stream>>>(cand, nq, n_keys, d_idx2, d_dist2, d_d2);
    ERP_LAUNCH(ctx, "bin_merge_kernel");

    set_knn_stats(ctx, ERP_ENGINE_TCGEN05_1X, true, n_seg, plan.units_per_cta, plan.grid, nullptr);
    return ERP_OK;
}

} // namespace erp
