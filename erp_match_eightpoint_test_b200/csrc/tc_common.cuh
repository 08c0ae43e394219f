// tc_common.cuh -- what the tcgen05 kernels share (knn_tc.cu and knn_tc1.cu: distances, knn_bin.cu: Hamming distances,
// score_tc.cu: residuals): inline-PTX wrappers (mbarrier, TMA, tcgen05 / TMEM), TMEM allocation, the tensor-map encoder,
// the stream-K planner and the launcher; and the query-pair pipeline (barriers, TMA producer, MMA ring walk, accumulator
// drain) that all four kernels run on.
#pragma once

#include "common.cuh"

#include <cuda.h>   // CUtensorMap (types only; the encoder is fetched through the runtime)

namespace erp {

constexpr int TC_SMEM_LIMIT = 232448;   // 227 KB of dynamic shared memory per CTA

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must surface as a launch failure, not as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    if (mbar_try_wait(bar, parity)) return;
    long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, 128 x 256 x 8, tf32 inputs, fp32 accumulate
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, 128 x 256 x 16, f16 inputs, fp32 accumulate: the same 32 bytes of every operand row as
// one tf32 instruction, at twice the rate
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, 128 x 256 x 32, s8 inputs, s32 accumulate
__device__ __forceinline__ void tc_mma_i8(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same with A read from tensor memory (lane = row, one tf32 per column): only B is fetched from shared memory
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// shared memory -> tensor memory, 128 rows x 32 bytes (8 columns) of the matrix a K-major descriptor names; asynchronous,
// ordered with the MMAs the same thread issues afterwards
__device__ __forceinline__ void tc_cp_128x256b(uint32_t taddr, uint64_t s_desc)
{
    asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(taddr), "l"(s_desc) : "memory");
}
// 32 lanes x 32 consecutive columns: thread i of the warp receives lane (base + i)
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// shared-memory matrix descriptor: K-major, 128-byte swizzle, rows of 128 bytes, 8-row groups of
// 1024 bytes (SBO), descriptor version 1 (sm_100).  addr may point inside the first swizzle row
// (k advance of 32 bytes per UMMA K step).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFF) >> 4);          // start address, bits [0,14)
    d |= (uint64_t)1 << 16;                          // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset, bits [32,46)
    d |= (uint64_t)1 << 46;                          // version
    d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
    return d;
}
// K-major rows of 32 bytes (ONE tf32 k step), 32-byte swizzle: 8-row groups are 256 bytes apart
__device__ __forceinline__ uint64_t smem_desc_sw32(uint32_t addr)
{
    uint64_t d = 0;
    d |= (uint64_t)((addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(256 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)6 << 61;                          // SWIZZLE_32B
    return d;
}
// wait for this thread's outstanding tcgen05.ld; the registers are operands so that no use of
// them can be scheduled above the wait
__device__ __forceinline__ void tc_wait_ld32(uint32_t (&v)[32])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                   "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                   "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
                 :
                 : "memory");
}

__device__ __forceinline__ void tc_ld8(uint32_t taddr, uint32_t (&v)[8])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tc_wait_ld8(uint32_t (&v)[8])
{
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7])
                 :
                 : "memory");
}

// all 512 TMEM columns (two accumulators of 256) for the CTA: the allocating warp writes their base address to *slot, and
// after the CTA barrier every thread returns it
__device__ __forceinline__ uint32_t tmem_alloc(bool alloc_warp, uint32_t* slot)
{
    if (alloc_warp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *slot;
}
// teardown: once every warp of the CTA is done with tensor memory, the allocating warp frees it
__device__ __forceinline__ void tmem_free(bool alloc_warp, uint32_t base)
{
    tc_fence_before();
    __syncthreads();
    if (alloc_warp) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(512) : "memory");
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn lookup_encode_fn()
{
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
        return reinterpret_cast<EncodeTiledFn>(p);
    cudaGetLastError();
    return nullptr;
}
inline EncodeTiledFn encode_fn()
{
    static const EncodeTiledFn fn = lookup_encode_fn();     // C++11 magic static: initialised once, thread safe
    return fn;
}

// rows x row_elems, row major, elements of type (esize bytes each); box = one 128-byte swizzle row (32 floats, 64 halves or
// 128 bytes) x box_rows, zero fill out of bounds; narrow = true: box = one 32-byte swizzle row x box_rows for the
// single-k-step operands
inline int make_map(CUtensorMap* map, const void* base, int rows, int row_elems, int box_rows, CUtensorMapDataType type, int esize,
                    bool narrow = false)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled is not available from this driver"); return ERP_E_CUDA; }
    cuuint64_t dims[2] = {(cuuint64_t)row_elems, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)row_elems * esize};
    cuuint32_t box[2] = {(narrow ? 32u : 128u) / esize, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, type, 2, const_cast<void*>(base), dims, strides,
                    box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, narrow ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return ERP_E_CUDA; }
    return ERP_OK;
}

// Stream-K plan: the n_rows x n_ttiles unit grid (row of query tiles major) is cut into equal contiguous ranges, one per
// CTA.  A row may be cut into at most max_seg segments (each writes its own candidate lists), which bounds the range
// length from below for small n_rows.
struct StreamK { int units_per_cta, n_seg, grid; };
inline StreamK stream_k_plan(int n_rows, int n_ttiles, int sms, int max_seg)
{
    const long total = (long)n_rows * n_ttiles;
    long L = (total + sms - 1) / sms;
    const long lmin = max_seg > 2 ? (n_ttiles + (max_seg - 2) - 1) / (max_seg - 2) : n_ttiles;   // <= max_seg-2 interior cuts + 1
    if (L < lmin) L = lmin;
    if (L < 1) L = 1;
    const long segs = (n_ttiles + L - 1) / L + 1;    // multiples of L strictly inside one row: at most (n_ttiles + L - 1) / L
    return {(int)L, (int)(segs > max_seg ? max_seg : segs), (int)((total + L - 1) / L)};
}

// sets the dynamic shared memory of Kernel once per device, launches it on the context's stream and checks the launch
template <auto Kernel, class... Args>
inline int launch_tc_kernel(erp_ctx* ctx, const char* name, int grid, int block, int smem, const Args&... args)
{
    static std::atomic<uint64_t> configured{0};
    ERP_TRY(ensure_dynamic_smem(ctx, Kernel, smem, configured));
    Kernel<<<grid, block, smem, ctx->stream>>>(args...);
    ERP_LAUNCH(ctx, name);
    return ERP_OK;
}


// Columns whose approximate score is above "2nd best so far + slack" can never be one of the exact two nearest neighbours
// (their exact distance exceeds the exact distance of the approximate runner-up): both distance kernels keep only columns
// below it.  slack = 2 * kappa * (|q|^2 + max|t|^2) for a score error of at most kappa * (|q|^2 + max|t|^2).
__device__ __forceinline__ float slack_of(float qn, float tn_max, float kappa)
{
    return __fmul_rn(__fmul_rn(2.0002f * kappa, __fadd_rn(qn, tn_max)), 1.0f);
}
// Candidate list of the one-product engine (knn_tc1.cu), 8 entries per (query row, list): [0], [1] = the two best scores so far in
// order (all the threshold needs), [2..7] = a FIFO of the other columns that were within the slack of the runner-up when
// they arrived (newest first).  An entry pushed out of the FIFO lowers floor_thr to its score (and with it the threshold),
// every other dropped column scored >= the threshold in force, so min(floor_thr, final threshold) bounds all
// non-candidates of the list.
// Scores carry their column (mod 8) in the three low mantissa bits -- the minimum of the packed keys is the winning
// score AND its position, which replaces a dynamic register index; the 2^-21 relative perturbation is part of the margin
// in F_KAPPA.  refine_kernel takes the list in any order.
//
// scan_chunk_lean: 32 accumulator columns of one query row, all in registers.  Common case: a min tree and ONE compare.
// Rare case (per lane, no TMEM access, no warp-wide vote): the groups of 8 columns whose minimum is below the threshold are
// selected out of the registers behind an opaque group id (so the compiler cannot specialise the code per group), packed,
// and inserted smallest first.  The threshold is also exchanged through shared memory with the thread that scans the other
// column range of the same row; any published value is a valid bound, so a lost race only costs pruning.
// The accumulator already holds |t|^2 - 2 q.t (the norm entered the MMA as an extra k step).
#if defined(ERP_TC_COUNTERS) && ERP_TC_COUNTERS == 2
static __device__ unsigned long long erp_evt[8];
#endif
__device__ __forceinline__ void scan_chunk_lean(const uint32_t (&v)[32], int col0, float slack, float (&bs)[8], int (&bi)[8],
                                                float* row_thr, float& floor_thr)
{
    const float other = *reinterpret_cast<volatile float*>(row_thr);
    float gm[4];
#pragma unroll
    for (int g = 0; g < 4; g++) {
        float s[8];
#pragma unroll
        for (int j = 0; j < 8; j++) s[j] = __uint_as_float(v[g * 8 + j]);
        gm[g] = fminf(fminf(fminf(s[0], s[1]), fminf(s[2], s[3])), fminf(fminf(s[4], s[5]), fminf(s[6], s[7])));
    }
    // floor_thr in the threshold is the capacity rule: once an entry has been pushed out, columns at or above its score
    // cannot improve the list's bound any more (all-equal scores would otherwise insert at every column)
    float thr = fminf(fminf(__fadd_rn(bs[1], slack), other), floor_thr);
    floor_thr = thr;
    if (fminf(fminf(gm[0], gm[1]), fminf(gm[2], gm[3])) < thr) {                                     // rare, per lane
        unsigned mine = (gm[0] < thr ? 1u : 0u) | (gm[1] < thr ? 2u : 0u) | (gm[2] < thr ? 4u : 0u) | (gm[3] < thr ? 8u : 0u);
#if defined(ERP_TC_COUNTERS) && ERP_TC_COUNTERS == 2
        const long long e0 = clock64();
        atomicAdd(&erp_evt[4], 1ull);
#endif
        do {
            int g = __ffs(mine) - 1;
            mine &= mine - 1;
            asm volatile("" : "+r"(g));
            const bool pl = (g & 1) != 0, ph = (g & 2) != 0;
#if defined(ERP_TC_COUNTERS) && ERP_TC_COUNTERS == 2
            atomicAdd(&erp_evt[5], 1ull);
#endif
            float k[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t lo = pl ? v[8 + j] : v[j], hi = pl ? v[24 + j] : v[16 + j];
                const uint32_t e = ph ? hi : lo;
                k[j] = __uint_as_float((e & ~7u) | (uint32_t)j);
            }
            const int cbase = col0 + g * 8;
            for (;;) {
                const float km = fminf(fminf(fminf(k[0], k[1]), fminf(k[2], k[3])), fminf(fminf(k[4], k[5]), fminf(k[6], k[7])));
                if (!(km < thr)) break;
#if defined(ERP_TC_COUNTERS) && ERP_TC_COUNTERS == 2
                atomicAdd(&erp_evt[6], 1ull);
#endif
                const int col = cbase + (int)(__float_as_uint(km) & 7u);
                // strict <: equal scores keep the earlier (lower) train index
                const bool lt0 = km < bs[0], lt1 = km < bs[1];
                const float pv = lt1 ? bs[1] : km;            // leaves the top two (or never enters)
                const int pi = lt1 ? bi[1] : col;
                bs[1] = lt0 ? bs[0] : (lt1 ? km : bs[1]);
                bi[1] = lt0 ? bi[0] : (lt1 ? col : bi[1]);
                bs[0] = lt0 ? km : bs[0];
                bi[0] = lt0 ? col : bi[0];
                thr = fminf(fminf(__fadd_rn(bs[1], slack), other), floor_thr);
                if (pv < thr) {
                    floor_thr = fminf(floor_thr, bs[7]);     // +inf while the FIFO has room
                    thr = fminf(thr, floor_thr);
#pragma unroll
                    for (int i = 7; i > 2; i--) { bs[i] = bs[i - 1]; bi[i] = bi[i - 1]; }
                    bs[2] = pv; bi[2] = pi;
                }
#pragma unroll
                for (int j = 0; j < 8; j++) k[j] = k[j] == km ? INFINITY : k[j];
            }
        } while (mine);
        if (thr < *reinterpret_cast<volatile float*>(row_thr)) *reinterpret_cast<volatile float*>(row_thr) = thr;
#if defined(ERP_TC_COUNTERS) && ERP_TC_COUNTERS == 2
        const long long e1 = clock64();
        {
            const unsigned am = __activemask();
            const bool warm = (col0 & 0xffff) < 4096;
            if ((threadIdx.x & 31) == __ffs(am) - 1) {
                atomicAdd(&erp_evt[warm ? 2 : 0], (unsigned long long)(e1 - e0));
                atomicAdd(&erp_evt[warm ? 3 : 1], 1ull);
            }
        }
#endif
    }
}

// A CTA's unit range cut into segments: consecutive train tiles of one query tile.  Host-callable so that
// tests/test_plan_host.py can check the plan's coverage and list slots without a GPU.
struct SegIter {
    long u, end;
    int n_ttiles, L;
    __host__ __device__ SegIter(int n_qtiles, int n_ttiles_, int units_per_cta, int cta)
    {
        L = units_per_cta; n_ttiles = n_ttiles_;
        u = (long)cta * L;
        long total = (long)n_qtiles * n_ttiles;
        end = u + L < total ? u + L : total;
    }
    // next segment: query tile, train tiles [t0, t1), list slot of the segment within its query tile
    __host__ __device__ bool next(int& qtile, int& t0, int& t1, int& seg)
    {
        if (u >= end) return false;
        qtile = (int)(u / n_ttiles);
        long row0 = (long)qtile * n_ttiles;
        t0 = (int)(u - row0);
        long rem = end - u;
        t1 = rem < n_ttiles - t0 ? t0 + (int)rem : n_ttiles;
        seg = (int)(u / L - row0 / L);      // CTA boundaries (multiples of L) in (row0, u]
        u += t1 - t0;
        return true;
    }
};

// Instrumented builds (scripts/build_variant.sh N): -DERP_TC_COUNTERS=1 adds clock64 phase timers to the MMA issuer and the
// epilogue warps of knn_tc1.cu, =2 counts and times the insert path (scan_chunk_lean); both print after every launch.  Off
// by default.
#ifndef ERP_TC_COUNTERS
#define ERP_TC_COUNTERS 0
#endif
#if ERP_TC_COUNTERS == 1
static __device__ unsigned long long erp_clk[8];
#define TCC_DECL unsigned long long lclk[6] = {0, 0, 0, 0, 0, 0}
#define TCC_CLOCK(name) const long long name = clock64()
#define TCC_ADD(i, v) (lclk[i] += (unsigned long long)(v))
#define TCC_FLUSH() do { if ((threadIdx.x & 31) == 0) for (int i_ = 0; i_ < 6; i_++) if (lclk[i_]) atomicAdd(&erp_clk[i_], lclk[i_]); } while (0)
#else
#define TCC_DECL
#define TCC_CLOCK(name)
#define TCC_ADD(i, v)
#define TCC_FLUSH()
#endif

// one 128-byte k chunk of a K-major operand pair as four instructions over 32 bytes of every row; acc = false: the first
// one overwrites the accumulator
template <auto Mma>
__device__ __forceinline__ void mma_chunk(uint32_t d_tmem, uint32_t a, uint32_t b, uint32_t idesc, bool acc)
{
#pragma unroll
    for (int k = 0; k < 4; k++) Mma(d_tmem, smem_desc_sw128(a + k * 32), smem_desc_sw128(b + k * 32), idesc, acc || k != 0);
}

// ---- the query-pair pipeline of the four tcgen05 kernels --------------------------------------------------------------
// knn_tc1.cu (f16) and knn_bin.cu (i8): four instructions per k chunk; score_tc.cu: one tf32 k chunk, hypothesis tiles
// double-buffered (QB = 2); knn_tc.cu (3xTF32): one sub-tile of 2 x KCH chunks, hi and lo interleaved, up to eight
// instructions per chunk.
// SUB resident query sub-tiles of BM rows share every train tile of BN rows.  A row is KCH k chunks of one 128-byte swizzle
// row (CK elements of the tensor maps).  The query sub-tiles sit in q_smem as [QB][SUB][KCH] chunks, loaded once per
// segment into buffer seg_n % QB; the train chunks pass through a ring of NS slots in t_smem, the KCH chunks of a train tile
// in consecutive slots.  The product of a sub-tile and a train tile goes to one of the two TMEM accumulators of BN columns,
// alternately.
// Barriers, N_BARS of them from the constructor's base: full / empty [NS] (chunk landed / read by the MMAs of the last
// sub-tile), qfull / qempty [QB] (query sub-tiles landed / no longer read), tfull / tempty [2] (accumulator ready /
// drained, one arrival per epilogue warp).
template <int SUB, int KCH, int NS, int BM, int BN, int CK, int QB = 1>
struct PairPipe {
    static constexpr int QCH = BM * 128, TCH = BN * 128;    // bytes of a k chunk of a query sub-tile and of a train tile
    static constexpr int N_BARS = 2 * NS + 2 * QB + 4;
    uint8_t* q_smem;
    uint8_t* t_smem;
    uint64_t *full, *empty, *qfull, *qempty, *tfull, *tempty;

    __device__ PairPipe(uint8_t* q, uint8_t* t, uint64_t* bars)
        : q_smem(q), t_smem(t), full(bars), empty(bars + NS), qfull(bars + 2 * NS), qempty(qfull + QB), tfull(qempty + QB),
          tempty(tfull + 2) {}

    // one thread, after the kernel's own barriers: the fence publishes those too
    __device__ __forceinline__ void init(int epi_warps) const
    {
        for (int i = 0; i < NS; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < QB; i++) { mbar_init(&qfull[i], 1); mbar_init(&qempty[i], 1); }
        for (int i = 0; i < 2; i++) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], epi_warps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    // TMA producer (one thread); train tile tt of the plan is row block tt + t_off of map_t
    __device__ __forceinline__ void produce(const CUtensorMap* map_q, const CUtensorMap* map_t, SegIter it, int t_off = 0) const
    {
        uint32_t slot = 0, ph = 0, seg_n = 0;
        int qp, t0, t1, seg;
        for (; it.next(qp, t0, t1, seg); seg_n++) {
            const uint32_t qb = seg_n % QB;
            mbar_wait(&qempty[qb], ((seg_n / QB) & 1) ^ 1);
            mbar_expect_tx(&qfull[qb], SUB * KCH * QCH);
#pragma unroll
            for (int sub = 0; sub < SUB; sub++)
#pragma unroll
                for (int c = 0; c < KCH; c++)
                    tma_load_2d(map_q, &qfull[qb], q_smem + ((qb * SUB + sub) * KCH + c) * QCH, c * CK, (qp * SUB + sub) * BM);
            for (int tt = t0 + t_off; tt < t1 + t_off; tt++) {
#pragma unroll
                for (int c = 0; c < KCH; c++) {
                    mbar_wait(&empty[slot], ph ^ 1);
                    mbar_expect_tx(&full[slot], TCH);
                    tma_load_2d(map_t, &full[slot], t_smem + slot * TCH, c * CK, tt * BN);
                    if (++slot == NS) { slot = 0; ph ^= 1; }
                }
            }
        }
    }

    // MMA issuer (one thread).  mma(d_tmem, q, c, b) issues the products of k chunk c: q is the shared-memory address of the
    // sub-tile's query chunks, b that of the train slot holding chunk c.  After the k chunks of a (sub-tile, train tile),
    // hook(sub, tt_n, d_tmem) may add to the accumulator before it is committed to the epilogue; tt_n counts the train
    // tiles of the CTA.
    template <class Mma, class Hook>
    __device__ __forceinline__ void issue(uint32_t tmem_base, SegIter it, Mma mma, Hook hook) const
    {
        TCC_DECL;
        uint32_t slot = 0, ph = 0, seg_n = 0, tile_n = 0;
        const uint32_t q_base = smem_u32(q_smem), t_base = smem_u32(t_smem);
        uint32_t tt_n = 0;
        int qp, t0, t1, seg;
        for (; it.next(qp, t0, t1, seg); seg_n++) {
            const uint32_t qb = seg_n % QB;
            mbar_wait(&qfull[qb], (seg_n / QB) & 1);
            for (int tt = t0; tt < t1; tt++, tt_n++) {
                const uint32_t s0 = slot, p0 = ph;
#pragma unroll
                for (int sub = 0; sub < SUB; sub++, tile_n++) {
                    const uint32_t acc = tile_n & 1;
                    TCC_CLOCK(m0);
                    mbar_wait(&tempty[acc], ((tile_n >> 1) & 1) ^ 1);
                    TCC_ADD(3, clock64() - m0); TCC_ADD(4, 1);
                    const uint32_t d_tmem = tmem_base + acc * BN;
                    const uint32_t q = q_base + (qb * SUB + sub) * KCH * QCH;
                    uint32_t sl = s0, pp = p0;
#pragma unroll
                    for (int c = 0; c < KCH; c++) {
                        TCC_CLOCK(f0);
                        if (sub == 0) mbar_wait(&full[sl], pp);
                        TCC_ADD(5, clock64() - f0);
                        tc_fence_after();
                        mma(d_tmem, q, c, t_base + sl * TCH);
                        if (sub == SUB - 1) tc_commit(&empty[sl]);
                        if (++sl == NS) { sl = 0; pp ^= 1; }
                    }
                    hook(sub, tt_n, d_tmem);
                    tc_commit(&tfull[acc]);
                    if (sub == SUB - 1) { slot = sl; ph = pp; }
                }
            }
            tc_commit(&qempty[qb]);
        }
        TCC_FLUSH();
    }

    // epilogue warp: its 128 columns of accumulator acc at taddr go to registers, and the accumulator is handed back before
    // they are examined, so a slow insert path delays this warp's next read, not the next MMA
    __device__ __forceinline__ void drain(uint32_t taddr, uint32_t acc, uint32_t (&va)[32], uint32_t (&vb)[32], uint32_t (&vc)[32],
                                          uint32_t (&vd)[32]) const
    {
        tc_ld32(taddr, va);
        tc_ld32(taddr + 32, vb);
        tc_ld32(taddr + 64, vc);
        tc_ld32(taddr + 96, vd);
        tc_wait_ld32(va);
        tc_wait_ld32(vb);
        tc_wait_ld32(vc);
        tc_wait_ld32(vd);
        tc_fence_before();
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(&tempty[acc]);
    }
};

} // namespace erp
