// score_tc.cu -- best-hypothesis search on the tensor cores.  The H x M residual matrix
//     res[h][c] = sum_k Eh[h][k] * (l_c (x) r_c)[k],  k = 0..8          (src/epipolar_tool.cpp:100-107)
// is a GEMM with a 9-long contraction.  One tcgen05 pass with K = 32 carries the three 3xTF32
// products at once:
//     A row (hypothesis)     = [ Eh_hi(9) | Eh_hi(9) | Eh_lo(9) | 0 x 5 ]
//     B row (correspondence) = [ K_hi(9)  | K_lo(9)  | K_hi(9)  | 0 x 5 ]      (128 bytes = one swizzle row)
// so a 128 x 256 tile of residuals costs four UMMA instructions and never leaves the SM.  The
// epilogue (one hypothesis row per thread, tcgen05.ld 32x32b) counts, per hypothesis,
//     c_hi = #{ |res| < tau + delta }  >=  the exact inlier count of the SIMT kernel / the oracle,
// where delta bounds |res_3xTF32 - res_fp32chain| (it scales with sqrt(2) * max|l||r|): two
// instructions per residual (FSET + FADD).  Then, exactly (score_kernel, score.cu):
//     L* = count of the hypothesis with the largest c_hi           (a lower bound of the best count)
//     winner = best exact count over { h : c_hi[h] >= L* }         (nothing outside can reach L*)
// so the packed best is bit-identical to scoring everything with the fp32 fma chain, at a fraction
// of the FP32-pipe work.
//
// Progressive pruning (exact): the bound is accumulated in three passes over the correspondences.
// Pass A covers the first 2048; its best-looking hypothesis is scored exactly -> L*.  Pass B extends
// every bound until a hypothesis that is still empty could no longer reach L* (about m - L*
// correspondences); hypotheses with  bound so far + correspondences not yet seen < L*  are dropped,
// and pass C finishes only the survivors (typically a few % of H).  All lengths stay on the device:
// the kernel reads its hypothesis count and correspondence-tile range from memory.
//
// Work is cut stream-K style over (pair of hypothesis tiles, correspondence tile) units -- each 32 KB
// correspondence tile that TMA brings in feeds two 128-row accumulators, which halves the L2 -> shared
// memory traffic per MMA (with one it was the limiter: tensor pipe 42 % active).  A pair cut between two
// CTAs adds its partial counts atomically.  Producer and MMA issuer are the query-pair pipeline of tc_common.cuh
// (PairPipe, the pair double-buffered); the counting epilogue keeps its own software pipeline.
#include "score_common.cuh"
#include "tc_common.cuh"

namespace erp {

constexpr int SM_ROWS = 128;                 // hypotheses per tile (UMMA M)
constexpr int SN_ROWS = 256;                 // correspondences per tile (UMMA N)
constexpr int SA_BYTES = SM_ROWS * 128;      // 16 KB
constexpr int SB_BYTES = SN_ROWS * 128;      // 32 KB
constexpr int S_SUB = 2;                     // hypothesis tiles that share every correspondence tile (halves the L2 -> smem feed)
constexpr int S_NSLOT = 5;                   // B ring
constexpr int S_EPI_GROUPS = 2;
constexpr int S_EPI_THREADS = S_EPI_GROUPS * 128;
constexpr int S_THREADS = 128 + S_EPI_THREADS;
constexpr int S_EPI_COLS = SN_ROWS / S_EPI_GROUPS;
constexpr int S_BARS = 256;                  // mbarriers, TMEM slot and the epilogue's threshold word
constexpr int S_SMEM = 2 * S_SUB * SA_BYTES + S_NSLOT * SB_BYTES + S_BARS;
static_assert(S_SMEM <= TC_SMEM_LIMIT, "shared memory budget");
constexpr uint32_t S_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(SN_ROWS >> 3) << 17) | ((uint32_t)(SM_ROWS >> 4) << 24);
// |res_tc - res_chain| <= S_KAPPA * sqrt(2) * max_c |l_c||r_c|: 3xTF32 (2^-20) + the chain's own
// rounding (9 * 2^-24) with a factor ~8 to spare
constexpr float S_KAPPA = 1.0f / 65536.0f;

// ---- operand preparation ---------------------------------------------------------------
// row i of Es = split scaled E of hypothesis i; also clears the two bound arrays and publishes pass A's shape
// (the minimal-sample solver does the same in its own epilogue, geometry.cu: min8_kernel)
__global__ void prep_e_kernel(const double* __restrict__ E, int H, float* __restrict__ Es /* H x 32 */, float big,
                              int32_t* __restrict__ upper /* 2 x H */, int32_t* __restrict__ w, const RowScale rs)
{
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h == 0) { w[W_DYN_A] = H; w[W_DYN_A + 1] = 0; w[W_DYN_A + 2] = w[W_N0]; w[W_DYN_A + 3] = w[W_M]; }
    if (h >= H) return;
    float e[9];
    scale_E(E + (size_t)h * 9, e);
    write_e_row(e, big, Es + (size_t)h * 32, row_gain(e, rs, w));
    upper[h] = 0; upper[(size_t)H + h] = 0;
}

__global__ void prep_k_kernel(const float4* __restrict__ l4, const float4* __restrict__ r4, int m_cap, const int32_t* __restrict__ m_dev,
                              float* __restrict__ Ks /* roundup(m_cap, 256) x 32 */, int32_t* __restrict__ w)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = dev_len(m_dev, m_cap);
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    prep_k_slot(c, m, c < m ? l4[c] : zero, c < m ? r4[c] : zero, Ks, w);
}

// ---- the scoring kernel ------------------------------------------------------------------
struct ScoreTcParams {
    float tau;
    float big;                    // 2^k applied to every A row: tau * big in [2^30, 2^31)
    const unsigned* kmax_bits;
    const int32_t* dyn;           // device: { hypotheses (rows of the A matrix), first correspondence tile, end tile, m }
    int32_t* upper;               // one counter per A row, zeroed by the caller: partial sums are added
};

// the launch's unit grid, read from device memory by every role
struct ScoreShape {
    int H, ct_begin, n_htiles, n_ctiles, units_per_cta, m;
    __device__ explicit ScoreShape(const ScoreTcParams& p)
    {
        H = p.dyn[0]; ct_begin = p.dyn[1]; m = p.dyn[3];
        n_ctiles = max(p.dyn[2] - ct_begin, 0);
        n_htiles = (H + SM_ROWS * S_SUB - 1) / (SM_ROWS * S_SUB);            // tile PAIRS
        long total = (long)n_htiles * n_ctiles;
        units_per_cta = (int)((total + gridDim.x - 1) / gridDim.x);
        if (units_per_cta < 1) units_per_cta = 1;
    }
};

// 32 residuals of one hypothesis row -> 1.0f per residual with |res| < thr, summed pairwise into two packed fp32x2
// accumulators (FADD2).  The indicator comes from two different pipes, alternating by pair, so that neither limits:
//   * FSET.BF.LT |res|, thr                    (ALU pipe, half rate)
//   * FADD.SAT thr, -|res|                     (FMA pipe): residuals and threshold arrive scaled by 2^k with thr * 2^k >= 2^30,
//     so thr - |res| is 0 or at least one ulp >= 128 and the saturation yields exactly 0 or 1 (NaN -> 0, like the compare)
// 1.5 instructions per residual over two pipes instead of 2 with the ALU pipe saturated.  Counts stay exact in fp32 up to 2^24.
__device__ __forceinline__ float ind_set(uint32_t bits, float thr)
{
    float r;
    asm("set.lt.f32.f32 %0, %1, %2;" : "=f"(r) : "f"(fabsf(__uint_as_float(bits))), "f"(thr));
    return r;
}
__device__ __forceinline__ float ind_sat(uint32_t bits, float thr)
{
    float r;
    asm("add.rn.sat.f32 %0, %1, %2;" : "=f"(r) : "f"(thr), "f"(-fabsf(__uint_as_float(bits))));
    return r;
}
__device__ __forceinline__ void add_pair(unsigned long long& acc, float a, float b)
{
    unsigned long long p;
    asm("mov.b64 %0, {%1, %2};" : "=l"(p) : "f"(a), "f"(b));
    asm("add.rn.f32x2 %0, %0, %1;" : "+l"(acc) : "l"(p));
}
__device__ __forceinline__ void count_chunk(const uint32_t (&v)[32], float hi, unsigned long long (&acc)[2])
{
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
        add_pair(acc[0], ind_sat(v[j], hi), ind_sat(v[j + 1], hi));
        add_pair(acc[1], ind_set(v[j + 2], hi), ind_set(v[j + 3], hi));
    }
}
__device__ __forceinline__ int pair_total(const unsigned long long (&acc)[2])
{
    float a, b, c, d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(acc[0]));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(c), "=f"(d) : "l"(acc[1]));
    return (int)((a + b) + (c + d));
}

__global__ void __launch_bounds__(S_THREADS, 1)
score_tc_kernel(const __grid_constant__ CUtensorMap map_e, const __grid_constant__ CUtensorMap map_k, const ScoreTcParams p)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    // [2 buffers][S_SUB] hypothesis tiles of one k chunk (32 floats), then the S_NSLOT correspondence slots
    using Pipe = PairPipe<S_SUB, 1, S_NSLOT, SM_ROWS, SN_ROWS, 32, 2>;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * S_SUB * SA_BYTES + S_NSLOT * SB_BYTES);
    const Pipe pipe(smem, smem + 2 * S_SUB * SA_BYTES, bars);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + Pipe::N_BARS);
    // the epilogue's threshold word, clear of the barriers and the TMEM slot
    constexpr int HI_SH = 192;
    static_assert(Pipe::N_BARS * 8 + 4 <= HI_SH && HI_SH + 4 <= S_BARS, "barrier block");

    // roles: warps 0..7 epilogue, then TMEM allocator, idle, TMA producer, MMA issuer.  The scheduler
    // favours the highest warp id among eligible warps: the two single-thread feeders sit on top so
    // that the issue-bound epilogue never delays a TMA or an MMA.
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int W_ALLOC = S_EPI_THREADS / 32, W_TMA = W_ALLOC + 2, W_MMA = W_ALLOC + 3;

    if (warp == W_TMA && lane == 0) { tma_prefetch_desc(&map_e); tma_prefetch_desc(&map_k); }
    if (warp == W_MMA && lane == 0) pipe.init(S_EPI_THREADS / 32);
    const uint32_t tmem_base = tmem_alloc(warp == W_ALLOC, tmem_slot);

    // the four feeder warps need few registers; the eight epilogue warps take them over (128 accumulator columns in flight)
    if (warp >= W_ALLOC) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;" ::: "memory");
    if (warp == W_TMA) {
        // ================================================================ TMA producer
        if (lane == 0) {
            const ScoreShape sh(p);
            pipe.produce(&map_e, &map_k, SegIter(sh.n_htiles, sh.n_ctiles, sh.units_per_cta, blockIdx.x), sh.ct_begin);
        }
    } else if (warp == W_MMA) {
        // ================================================================ MMA issuer
        if (lane == 0) {
            const ScoreShape sh(p);
            pipe.issue(tmem_base, SegIter(sh.n_htiles, sh.n_ctiles, sh.units_per_cta, blockIdx.x),
                       [](uint32_t d_tmem, uint32_t a, int, uint32_t b) { mma_chunk<tc_mma_tf32>(d_tmem, a, b, S_IDESC, false); },
                       [](int, uint32_t, uint32_t) {});
        }
    }
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 224;" ::: "memory");
        // ================================================================ epilogue
        const int ew = warp & 3, cg = warp >> 2;
        const int row = ew * 32 + lane;
        // band around tau inside which the tensor-core value cannot decide the test
        const float kmax = __uint_as_float(*p.kmax_bits);
        const float delta = S_KAPPA * 1.41421356f * kmax;
        float hi = (p.tau + delta) * p.big;                             // the A operand carries the factor p.big (a power of two)
        if (!(delta < INFINITY)) hi = INFINITY;                         // non-finite input: every finite residual may be an inlier
        // the threshold is re-read (volatile) after every hand-back of an accumulator: the counting depends on that load, so
        // the assembler cannot sink the TMEM loads into the counting code and delay the hand-back
        volatile float* hi_sh = reinterpret_cast<volatile float*>(reinterpret_cast<uint8_t*>(bars) + HI_SH);
        *hi_sh = hi;
        uint32_t tile_n = 0;
        const ScoreShape sh(p);
        SegIter it(sh.n_htiles, sh.n_ctiles, sh.units_per_cta, blockIdx.x);
        int ht, c0, c1, seg;
        while (it.next(ht, c0, c1, seg)) {
            c0 += sh.ct_begin; c1 += sh.ct_begin;
            unsigned long long acc4[S_SUB][2];
#pragma unroll
            for (int sub = 0; sub < S_SUB; sub++) acc4[sub][0] = acc4[sub][1] = 0ull;
            int pad_total = 0;
            // Software pipeline over the tiles of the segment: while a tile is counted out of registers, the next tile's
            // accumulator is read into the buffers that have just been consumed (first two chunks after the first half of
            // the counting, the other two after the second half) and handed back -- the TMEM read latency and the wait
            // for the MMA hide behind the counting instead of adding to it.
            static_assert(S_EPI_COLS == 128 && S_SUB == 2, "four chunks of 32 columns per warp and tile, two tiles per round");
            uint32_t va[32], vb[32], vc[32], vd[32];
            const uint32_t lane_base = tmem_base + ((uint32_t)(ew * 32) << 16) + cg * S_EPI_COLS;
            if (c0 < c1) {
                const uint32_t acc = tile_n & 1;
                mbar_wait(&pipe.tfull[acc], (tile_n >> 1) & 1);
                tc_fence_after();
                const uint32_t taddr = lane_base + acc * SN_ROWS;
                tc_ld32(taddr, va); tc_ld32(taddr + 32, vb); tc_ld32(taddr + 64, vc); tc_ld32(taddr + 96, vd);
                tc_wait_ld32(va); tc_wait_ld32(vb); tc_wait_ld32(vc); tc_wait_ld32(vd);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&pipe.tempty[acc]);
                tile_n++;
            }
            for (int ct = c0; ct < c1; ct++) {
                const int colbase = ct * SN_ROWS + cg * S_EPI_COLS;
#pragma unroll
                for (int sub = 0; sub < S_SUB; sub++) {
                    // registers hold tile (ct, sub); tile_n already names the next one
                    const bool has_next = sub + 1 < S_SUB || ct + 1 < c1;
                    const uint32_t acc = tile_n & 1;
                    const uint32_t taddr = lane_base + acc * SN_ROWS;
                    const float hv = *hi_sh;
                    count_chunk(va, hv, acc4[sub]);
                    count_chunk(vb, hv, acc4[sub]);
                    if (has_next) {
                        mbar_wait(&pipe.tfull[acc], (tile_n >> 1) & 1);
                        tc_fence_after();
                        tc_ld32(taddr, va); tc_ld32(taddr + 32, vb);
                    }
                    count_chunk(vc, hv, acc4[sub]);
                    count_chunk(vd, hv, acc4[sub]);
                    if (has_next) {
                        tc_ld32(taddr + 64, vc); tc_ld32(taddr + 96, vd);
                        tc_wait_ld32(va); tc_wait_ld32(vb); tc_wait_ld32(vc); tc_wait_ld32(vd);
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&pipe.tempty[acc]);
                        tile_n++;
                    }
                }
                // zero-filled columns past m have res = 0 exactly and were counted -- unless the hypothesis row is NaN
                // (a sample with non-finite bearings): then nothing was counted, see the clamp below
                pad_total += S_EPI_COLS - min(max(sh.m - colbase, 0), S_EPI_COLS);
            }
#pragma unroll
            for (int sub = 0; sub < S_SUB; sub++) {
                const int h = (ht * S_SUB + sub) * SM_ROWS + row;
                if (h < sh.H) {
                    int n = pair_total(acc4[sub]);
                    if (0.f < hi) n = max(n - pad_total, 0);     // a finite row counted its pads: n >= pad_total
                    if (n) atomicAdd(p.upper + h, n);
                }
            }
        }
    }

    tmem_free(warp == W_ALLOC, tmem_base);
}

// ---- the small kernels between the passes ------------------------------------------------------
// After pass A: L* = a lower bound of the best exact count.  ANY hypothesis' exact count is one; the best-looking
// hypotheses give the tightest.  Every block scores the hypothesis with the largest bound among its own (1024 threads,
// ~50 correspondences each, four in flight) exactly over ALL correspondences -- the globally best-looking one is among
// them, so L* is at least what scoring that one alone would give -- and merges its packed (count, ~id) into *best
// like any other exact count.  The last block to finish takes the maximum and plans passes B and C.
constexpr int AP_THREADS = 1024;
template <int METRIC>
__global__ void __launch_bounds__(AP_THREADS)
argmax_plan_kernel(const int32_t* __restrict__ upper, const double* __restrict__ E, const float4* __restrict__ l4,
                   const float4* __restrict__ r4, float tau, float tau2, float sin2, unsigned long long hyp0, int32_t* __restrict__ w,
                   unsigned long long* __restrict__ best, int slack_div, int slack_tiles)
{
    __shared__ unsigned long long wbest[AP_THREADS / 32];
    __shared__ int wsum[AP_THREADS / 32];
    __shared__ float Es[9];
    __shared__ int first_sh, last;
    const int H = w[W_DYN_A], lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int m = w[W_M];
    unsigned long long b = 0;
    for (int h = blockIdx.x * AP_THREADS + threadIdx.x; h < H; h += gridDim.x * AP_THREADS) {
        unsigned long long v = ((unsigned long long)(uint32_t)upper[h] << 32) | (uint32_t)(0xFFFFFFFFu - (uint32_t)h);
        b = v > b ? v : b;
    }
    for (int o = 16; o > 0; o >>= 1) { unsigned long long y = __shfl_down_sync(0xffffffffu, b, o); b = y > b ? y : b; }
    if (lane == 0) wbest[wid] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < AP_THREADS / 32; i++) b = wbest[i] > b ? wbest[i] : b;
        // a block whose range is empty (H < its first index) has nothing to score
        first_sh = b ? (int)(0xFFFFFFFFu - (uint32_t)(b & 0xFFFFFFFFull)) : -1;
        if (first_sh >= 0) scale_E(E + (size_t)first_sh * 9, Es);
    }
    __syncthreads();
    const int first = first_sh;
    int cnt = 0;
    if (first >= 0) {
        float e[9];
#pragma unroll
        for (int i = 0; i < 9; i++) e[i] = Es[i];
        // four correspondences in flight per thread: the loop is a chain of L2 round trips otherwise
        for (int c = threadIdx.x; c < m; c += 4 * AP_THREADS) {
            float4 l[4], r[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int cu = c + u * AP_THREADS;
                l[u] = cu < m ? l4[cu] : make_float4(0.f, 0.f, 0.f, 0.f);
                r[u] = cu < m ? r4[cu] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                float k[9];
                kron9(l[u], r[u], k);
                cnt += (c + u * AP_THREADS < m && inlier<METRIC>(e, k, l[u], r[u], tau, tau2, sin2)) ? 1 : 0;
            }
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) wsum[wid] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int exact = 0;
        for (int i = 0; i < AP_THREADS / 32; i++) exact += wsum[i];
        if (first >= 0) {
            atomicMax(best, ((unsigned long long)(uint32_t)exact << 32) | (uint32_t)(0xFFFFFFFFu - (uint32_t)(hyp0 + (unsigned long long)first)));
            atomicMax(w + W_LSTAR, exact);
        }
        __threadfence();
        last = atomicAdd(w + W_DONE, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!last || threadIdx.x != 0) return;
    __threadfence();
    const int lstar = *reinterpret_cast<volatile int32_t*>(w + W_LSTAR);
    // pass B extends the bounds to tile ct1: far enough that a hypothesis with nothing so far can no longer reach L*
    // (correspondences a discarded hypothesis may still be missing: m - seen < L*  <=>  seen > m - L*)
    const int n0 = w[W_N0], n_ct = w[W_NCT];
    long need = (long)m - lstar;
    need += need / slack_div + slack_tiles * SN_ROWS;       // slack: bad hypotheses still collect a few inliers
    int ct1 = (int)((need + SN_ROWS - 1) / SN_ROWS);
    if (ct1 < n0) ct1 = n0;
    if (ct1 > n_ct || lstar * 4 < m) ct1 = n_ct;           // weak best model: pruning cannot pay, finish in pass B
    w[W_DYN_B] = H; w[W_DYN_B + 1] = n0; w[W_DYN_B + 2] = ct1; w[W_DYN_B + 3] = m;
    w[W_DYN_C] = 0; w[W_DYN_C + 1] = ct1; w[W_DYN_C + 2] = n_ct; w[W_DYN_C + 3] = m;   // [0] = survivors, counted by the select kernel
    const long seen = (long)ct1 * SN_ROWS;
    w[W_REMAIN] = seen >= m ? 0 : (int)(m - seen);
}

// survivors of pass B: bound so far + correspondences not yet seen >= L*.  A survivor's operand row moves to its slot
// of the pass-C matrix right here.  One atomic per block (the per-warp version spent its 24 us on ~27k atomics to one word).
__global__ void __launch_bounds__(256)
survivor_select_kernel(const int32_t* __restrict__ upper, int32_t* __restrict__ w, int32_t* __restrict__ list,
                       const float4* __restrict__ Es, float4* __restrict__ Es2)
{
    __shared__ int wcount[8], wbase[8];
    const int H = w[W_DYN_A];
    const int h = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const bool keep = h < H && upper[h] + w[W_REMAIN] >= w[W_LSTAR] && w[W_REMAIN] > 0;
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) wcount[wid] = __popc(bal);
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
        for (int i = 0; i < 8; i++) { wbase[i] = total; total += wcount[i]; }
        const int base = total ? atomicAdd(&w[W_DYN_C], total) : 0;
        for (int i = 0; i < 8; i++) wbase[i] += base;
    }
    __syncthreads();
    if (keep) {
        const int s = wbase[wid] + __popc(bal & ((1u << lane) - 1));
        list[s] = h;
#pragma unroll
        for (int i = 0; i < 8; i++) Es2[(size_t)s * 8 + i] = Es[(size_t)h * 8 + i];
    }
}

// contenders: hypotheses whose completed bound still reaches L*.  With nothing left for pass C (REMAIN == 0) every
// hypothesis is complete after pass B and the survivor list is empty.
__global__ void final_select_kernel(const int32_t* __restrict__ upper, const int32_t* __restrict__ upper2,
                                    const int32_t* __restrict__ survivors, int32_t* __restrict__ w, int32_t* __restrict__ list)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const bool direct = w[W_REMAIN] == 0;
    const int n = direct ? w[W_DYN_A] : w[W_DYN_C];
    const int h = s < n ? (direct ? s : survivors[s]) : -1;
    const bool keep = h >= 0 && upper[h] + (direct ? 0 : upper2[s]) >= w[W_LSTAR];
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (!bal) return;
    int lane = threadIdx.x & 31, base = 0;
    if (lane == 0) base = atomicAdd(&w[W_LENF], __popc(bal));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (keep) list[base + __popc(bal & ((1u << lane) - 1))] = h;
}

bool score_tc_preferred(int H, int m) { return (double)H * (double)m >= 3.0e7 && m >= 1 && m < (1 << 24) && H >= 1; }

static int launch_score_tc(erp_ctx* ctx, const CUtensorMap& me, const CUtensorMap& mk, const ScoreTcParams& p)
{
    cudaEvent_t e0, e1;
    ERP_TRY(score_event(ctx, &e0));
    ERP_TRY(launch_tc_kernel<score_tc_kernel>(ctx, "score_tc_kernel", ctx->sm_count, S_THREADS, S_SMEM, me, mk, p));
    ERP_TRY(score_event(ctx, &e1));
    return ERP_OK;
}

// power-of-two factor on the hypothesis operand: the scaled threshold lies in [2^30, 2^31) (see count_chunk)
float score_tc_big(float tau)
{
    int ex = 0;
    frexpf(tau > 1e-30f ? tau : 1e-30f, &ex);            // tau = f * 2^ex, f in [0.5, 1)
    return ldexpf(1.0f, 31 - ex);
}

// scratch of one search: operand matrices, bound arrays, lists, device words
int score_tc_buffers(erp_ctx* ctx, int H, int m_cap, ScoreTcBuffers* b)
{
    int st = ERP_OK;
    b->Es = ctx->scratch<float>(S_SC_E, (size_t)H * 32, &st);
    b->Es2 = ctx->scratch<float>(S_SC_E2, (size_t)H * 32, &st);
    b->Ks = ctx->scratch<float>(S_SC_K, (size_t)cdiv(m_cap, SC_TILE) * SC_TILE * 32, &st);
    b->w = ctx->scratch<int32_t>(S_SC_MISC, W_WORDS, &st);
    b->upper = ctx->scratch<int32_t>(S_SC_BOUNDS, (size_t)H * 2, &st);       // [H] all hypotheses, [H] pass C rows
    b->list = ctx->scratch<int32_t>(S_SC_LIST, (size_t)H * 2, &st);          // [H] survivors, [H] contenders
    return st;
}

// the correspondence side, once per call (all hypothesis chunks share it)
int score_tc_prepare(erp_ctx* ctx, const ScoreTcBuffers& b, const float* d_l4, const float* d_r4, int m_cap, const int32_t* d_m)
{
    if (m_cap >= (1 << 24)) { set_error("score_tc: more than 2^24 correspondences"); return ERP_E_LIMIT; }
    ERP_CUDA(cudaMemsetAsync(b.w, 0, W_WORDS * sizeof(int32_t), ctx->stream));
    prep_k_kernel<<<cdiv(m_cap, 256), 256, 0, ctx->stream>>>((const float4*)d_l4, (const float4*)d_r4, m_cap, d_m, b.Ks, b.w);
    ERP_LAUNCH(ctx, "prep_k_kernel");
    return ERP_OK;
}

// merges into *d_best the packed (count << 32 | ~id) of the best of the H hypotheses, exactly as
// erp_score_dev + best_kernel would (algebraic residual).  The correspondence operand and the m-dependent words are
// in place (score_tc_prepare, or the fused gather of geometry.cu) and the per-chunk words are clear; es_ready: the
// hypothesis operand and the cleared bounds are in place too (min8_kernel wrote them).
int score_tc_search(erp_ctx* ctx, const ScoreTcBuffers& b, const double* d_E, int H, const float* d_l4, const float* d_r4, int m_cap,
                    int metric, float tau, uint64_t hyp0, bool es_ready, int32_t* d_counts_scratch, uint64_t* d_best)
{
    const float big = score_tc_big(tau);
    const double sd = sin((double)tau);
    const float tau2 = tau * tau, sin2 = (float)(sd * sd);
    RowScale rs;
    rs.metric = metric; rs.tau = tau; rs.sin_tau = (float)sd;
    int32_t* w = b.w;
    int32_t *upper = b.upper, *upper2 = b.upper + H, *survivors = b.list, *contenders = b.list + H;
    if (!es_ready) {
        prep_e_kernel<<<cdiv(H, 256), 256, 0, ctx->stream>>>(d_E, H, b.Es, big, upper, w, rs);
        ERP_LAUNCH(ctx, "prep_e_kernel");
    }
    CUtensorMap me, me2, mk;
    ERP_TRY(make_map(&me, b.Es, H, 32, SM_ROWS, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4));
    ERP_TRY(make_map(&me2, b.Es2, H, 32, SM_ROWS, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4));
    ERP_TRY(make_map(&mk, b.Ks, m_cap, 32, SN_ROWS, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4));
    ScoreTcParams p;
    p.tau = tau; p.big = big; p.kmax_bits = (const unsigned*)(w + W_KMAX);

    // pass A: every hypothesis, the first n0 correspondence tiles
    p.dyn = w + W_DYN_A; p.upper = upper;
    ERP_TRY(launch_score_tc(ctx, me, mk, p));
    {
        const int grid = min(cdiv(H, AP_THREADS), ctx->sm_count);
        static const int slack_div = [] { const char* e = getenv("ERP_B200_PRUNE_DIV"); return e && atoi(e) > 0 ? atoi(e) : 16; }();
        static const int slack_tiles = [] { const char* e = getenv("ERP_B200_PRUNE_TILES"); return e ? atoi(e) : 2; }();
        const float4 *l4 = (const float4*)d_l4, *r4 = (const float4*)d_r4;
        unsigned long long* bp = (unsigned long long*)d_best;
        if (metric == ERP_METRIC_ALGEBRAIC) argmax_plan_kernel<ERP_METRIC_ALGEBRAIC><<<grid, AP_THREADS, 0, ctx->stream>>>(upper, d_E, l4, r4, tau, tau2, sin2, hyp0, w, bp, slack_div, slack_tiles);
        else if (metric == ERP_METRIC_SAMPSON) argmax_plan_kernel<ERP_METRIC_SAMPSON><<<grid, AP_THREADS, 0, ctx->stream>>>(upper, d_E, l4, r4, tau, tau2, sin2, hyp0, w, bp, slack_div, slack_tiles);
        else argmax_plan_kernel<ERP_METRIC_ANGULAR><<<grid, AP_THREADS, 0, ctx->stream>>>(upper, d_E, l4, r4, tau, tau2, sin2, hyp0, w, bp, slack_div, slack_tiles);
        ERP_LAUNCH(ctx, "argmax_plan_kernel");
    }
    // pass B: every hypothesis, tiles [n0, ct1)
    p.dyn = w + W_DYN_B;
    ERP_TRY(launch_score_tc(ctx, me, mk, p));
    survivor_select_kernel<<<cdiv(H, 256), 256, 0, ctx->stream>>>(upper, w, survivors, (const float4*)b.Es, (float4*)b.Es2);
    ERP_LAUNCH(ctx, "survivor_select_kernel");
    // pass C: the survivors, tiles [ct1, n_ct)
    p.dyn = w + W_DYN_C; p.upper = upper2;
    ERP_TRY(launch_score_tc(ctx, me2, mk, p));
    final_select_kernel<<<cdiv(H, 256), 256, 0, ctx->stream>>>(upper, upper2, survivors, w, contenders);
    ERP_LAUNCH(ctx, "final_select_kernel");
    ctx->sc_misc_dev = w;
    return score_list_best(ctx, d_E, H, contenders, w + W_LENF, d_l4, d_r4, m_cap, w + W_M, metric, tau, hyp0, d_counts_scratch, d_best);
}

} // namespace erp
