// common.cuh -- context, error plumbing and scratch management shared by the .cu files.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <functional>
#include <string>
#include <vector>

#include "erp_b200.h"

#define ERP_API extern "C" __attribute__((visibility("default")))

namespace erp {

void set_error(const char* fmt, ...);

#define ERP_CUDA(call)                                                                   \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            erp::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return ERP_E_CUDA;                                                           \
        }                                                                                \
    } while (0)

#define ERP_TRY(call)                 \
    do {                              \
        int s_ = (call);              \
        if (s_ != ERP_OK) return s_;  \
    } while (0)

#define ERP_ARG(cond, code, ...)       \
    do {                               \
        if (!(cond)) {                 \
            erp::set_error(__VA_ARGS__); \
            return (code);             \
        }                              \
    } while (0)

// grow-only device / pinned-host buffer
struct Buf {
    void* p = nullptr;
    size_t cap = 0;
    bool host = false;
    int reserve(size_t bytes);
    void release();
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

enum ScratchId {
    S_Q = 0, S_T, S_IDX2, S_DIST2, S_D2, S_REVQ, S_REVD2, S_OUT, S_NOUT, S_BLOCKCNT,
    S_L3, S_R3, S_L4, S_R4, S_XY, S_SAMPLES, S_GRAM, S_E, S_EF, S_POSE, S_COUNTS, S_PACKED,
    S_MASK, S_PARTIAL, S_CONS, S_MISC,
    S_TC_Q, S_TC_T, S_TC_QN, S_TC_TN, S_TC_CAND, S_TC_LIST, S_TC_MISC,
    S_RS_IDX, S_RS_DIST, S_RS_D2, S_RS_PARTIAL,
    S_SC_E, S_SC_E2, S_SC_K, S_SC_MISC, S_SC_BOUNDS, S_SC_LIST,
    S_IMG_IN, S_IMG_OUT, S_RESULT, S_GATHER, S_XCHG, S_TC_ROWTHR,
    S_COUNT_
};

} // namespace erp

namespace erp { struct Comm; struct GraphCache; struct StagePool; }

struct erp_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;             // host-buffer calls upload query chunks here while the previous chunk computes
    cudaEvent_t ev_copy[10] = {};                   // "chunk c is on the device" (0..6), fork events (7: chunked upload, 8: staged upload), 9: keypoints of a host pair call
    int tc_chunk = 0;                               // > 0: later query chunk of one host call: train operand and statistics carry over
    int engine = ERP_ENGINE_AUTO;
    uint64_t launches = 0;
    int64_t knn_stats[5] = {0, 0, 0, 0, 0};
    bool knn_bin = false;                           // the last erp_knn2* search was on binary descriptors (knn_bin.cu)
    int32_t* sc_misc_dev = nullptr;                 // device words of the last tensor-core best search: ., max c_lo, list length
    int32_t* tc_misc_dev = nullptr;                 // device words of the last tcgen05 call: re-scan count, ., deviation
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;   // around the dominant distance kernel
    cudaEvent_t ev_stage[4] = {};                   // one pair: start, matches filtered, correspondences gathered, pose done
    erp::Comm* comm = nullptr;                      // multi-GPU: this context's rank of an NCCL clique (dist.cu)
    // CUDA graph of the last device-resident pair call (api.cu: graph_run): the second identical call is captured,
    // later ones are one cudaGraphLaunch.  scratch_gen counts scratch re-allocations (a cached graph holds pointers).
    bool capturing = false;
    uint64_t scratch_gen = 0;
    erp::GraphCache* graph = nullptr;
    erp::StagePool* stage = nullptr;                // pinned staging of pageable host buffers (api.cu: upload_rows)
    std::vector<cudaEvent_t> ev_score;              // pairs around the scoring kernel launches of the last RANSAC call
    int n_ev_score = 0;                             // events used by that call
    erp::Buf dev[erp::S_COUNT_];
    erp::Buf pinned[8];

    template <class T> T* scratch(int id, size_t count, int* status) {
        void* before = dev[id].p;
        int s = dev[id].reserve(count * sizeof(T));
        if (s != ERP_OK) *status = s;
        if (dev[id].p != before) scratch_gen++;
        return dev[id].as<T>();
    }
    template <class T> T* host_scratch(int id, size_t count, int* status) {
        pinned[id].host = true;
        int s = pinned[id].reserve(count * sizeof(T));
        if (s != ERP_OK) *status = s;
        return pinned[id].as<T>();
    }
};

namespace erp {

inline int check_launch(erp_ctx* ctx, const char* what)
{
    ctx->launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
        return ERP_E_CUDA;
    }
    return ERP_OK;
}

#define ERP_LAUNCH(ctx, name) ERP_TRY(erp::check_launch((ctx), (name)))

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

inline int cdiv(int a, int b) { return (a + b - 1) / b; }

#ifdef __CUDACC__
__device__ __forceinline__ float tf32_rna(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}
// a length that lives on the device (the match count) capped by the capacity the launch was sized for
__device__ __forceinline__ int dev_len(const int32_t* __restrict__ n_dev, int cap)
{
    if (!n_dev) return cap;
    const int n = *n_dev;
    return n < 0 ? 0 : (n < cap ? n : cap);
}
#endif

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: one bit per device ordinal and kernel
// (a process may hold contexts on several GPUs).  Setting it twice is harmless, so the flag needs no lock.
template <class Kernel>
inline int ensure_dynamic_smem(erp_ctx* ctx, Kernel kernel, int bytes, std::atomic<uint64_t>& done)
{
    const uint64_t bit = 1ull << (ctx->device & 63);
    if (done.load(std::memory_order_acquire) & bit) return ERP_OK;
    ERP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done.fetch_or(bit, std::memory_order_release);
    return ERP_OK;
}

// what erp_ctx_last_knn_stats and erp_ctx_last_knn_operands report about the last search: engine, binary rows, segments per
// query row, units per CTA, grid; misc = the device words of a tcgen05 search that has a re-scan (its count is read from
// there: knn_stats[1] = -1), null otherwise (nothing re-scanned: 0)
inline void set_knn_stats(erp_ctx* ctx, int engine, bool bin, int n_seg, int units_per_cta, int grid, int32_t* misc)
{
    ctx->knn_stats[0] = engine;
    ctx->knn_stats[1] = misc ? -1 : 0;
    ctx->knn_stats[2] = n_seg;
    ctx->knn_stats[3] = units_per_cta;
    ctx->knn_stats[4] = grid;
    ctx->knn_bin = bin;
    ctx->tc_misc_dev = misc;
}

// timing events are recorded by the library on its own stream; inside a stream capture they become external event-record
// nodes, so a replayed graph refreshes them like a direct call does
inline cudaError_t record_timing(erp_ctx* ctx, cudaEvent_t ev)
{
    return cudaEventRecordWithFlags(ev, ctx->stream, ctx->capturing ? cudaEventRecordExternal : cudaEventRecordDefault);
}

// next event of the scoring-kernel timer (created on demand, reused across calls)
inline int score_event(erp_ctx* ctx, cudaEvent_t* ev)
{
    if (ctx->n_ev_score == (int)ctx->ev_score.size()) {
        cudaEvent_t e;
        ERP_CUDA(cudaEventCreate(&e));
        ctx->ev_score.push_back(e);
    }
    *ev = ctx->ev_score[ctx->n_ev_score++];
    ERP_CUDA(record_timing(ctx, *ev));
    return ERP_OK;
}

// ---- internal device-level entry points shared across translation units ----
int knn2_exact(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
               const int32_t* d_qlist, int nlist, int idx_offset,
               int32_t* d_idx2, float* d_dist2, double* d_d2);
int knn2_tc(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
            int32_t* d_idx2, float* d_dist2, double* d_d2);
bool knn2_tc_supported(int nq, int nt, int dim);
bool knn2_tc_preferred(int nq, int nt, int dim);
int knn2_tc1(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
             int32_t* d_idx2, float* d_dist2, double* d_d2);
bool knn2_bin_preferred(int nq, int nt);
int knn2_bin(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes, bool tc,
             int32_t* d_idx2, float* d_dist2, double* d_d2);
int near_ties(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim, const int32_t* d_idx2, const double* d_d2,
              double rel_tol, int32_t* d_third, uint8_t* d_flags);
int tc_misc_begin(erp_ctx* ctx, int32_t* misc);
int tc_misc_end(erp_ctx* ctx, int32_t* misc);
int refine_launch(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim, int n_lists, int topk, double kappa,
                  double f16_abs, const int32_t* cand, const float* cand_s, const float* cand_thr, unsigned* misc, int32_t* d_idx2, float* d_dist2,
                  double* d_d2, int32_t* rescan_list);
int knn2_exact_rescan(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                      const int32_t* d_list, const int32_t* d_count, int max_rows,
                      int32_t* d_idx2, float* d_dist2, double* d_d2);
// ---- RANSAC chain (score.cu, score_tc.cu, geometry.cu): every length that depends on the match count is read from
// device memory (d_m, capped by m_cap, the size the launches are made for), so nothing between the matcher and the
// final result copy waits for the host
constexpr int RANSAC_CHUNK = 1 << 20;
struct ScoreTcBuffers { float *Es, *Es2, *Ks; int32_t *w, *upper, *list; };
struct Min8Fused { float* Es = nullptr; float big = 0.f; int32_t* upper = nullptr; int32_t* w = nullptr; int metric = 0; float tau = 0.f, sin_tau = 0.f; };
int score_tc_buffers(erp_ctx* ctx, int H, int m_cap, ScoreTcBuffers* b);
int score_tc_prepare(erp_ctx* ctx, const ScoreTcBuffers& b, const float* d_l4, const float* d_r4, int m_cap, const int32_t* d_m);
int score_tc_search(erp_ctx* ctx, const ScoreTcBuffers& b, const double* d_E, int H, const float* d_l4, const float* d_r4, int m_cap,
                    int metric, float tau, uint64_t hyp0, bool es_ready, int32_t* d_counts_scratch, uint64_t* d_best);
float score_tc_big(float tau);
int score_list_best(erp_ctx* ctx, const double* d_E, int H_max, const int32_t* d_list, const int32_t* d_len,
                    const float* d_l4, const float* d_r4, int m_cap, const int32_t* d_m, int metric, float tau, uint64_t hyp0,
                    int32_t* d_counts, uint64_t* d_best);
bool score_tc_preferred(int H, int m);
bool ransac_uses_tc(erp_ctx* ctx, int H, int m_cap, int metric);
int ransac_search(erp_ctx* ctx, const double* d_l3, const double* d_r3, const float* d_l4, const float* d_r4, int m_cap,
                  const int32_t* d_m, uint64_t seed, uint64_t hyp_offset, int H, int S, int metric, float tau, bool k_ready,
                  uint64_t* d_packed);
int ransac_finish(erp_ctx* ctx, const double* d_l3, const double* d_r3, const float* d_l4, const float* d_r4, int m_cap,
                  const int32_t* d_m, uint64_t seed, const uint64_t* d_packed, int S, int metric, float tau,
                  uint8_t* d_mask, erp_ransac_result* d_result);
struct PoseBuffers { double *l3, *r3; float *l4, *r4; uint8_t* mask; erp_ransac_result* res; };
constexpr size_t W_WORDS_BYTES = 28 * sizeof(int32_t);     // == W_WORDS (score_common.cuh)
int pose_chain_buffers(erp_ctx* ctx, int m_cap, PoseBuffers* b);
int pose_chain_tail(erp_ctx* ctx, const double* dl, const double* dr, const float* dl4, const float* dr4, int m_cap, const int32_t* d_m,
                    uint64_t seed, uint64_t hyp_offset, int H, int S, int metric, float tau, bool k_ready, bool reduce,
                    uint8_t* d_mask, erp_ransac_result* d_res);
// ---- host entry points (api.cu): one implementation serves float and binary descriptors
// A descriptor kind: float rows of `dim` values (L2) or binary rows of `dim` bytes (Hamming).
struct RowKind {
    bool bin;
    int dim;
    static RowKind f32(int dim) { return {false, dim}; }
    static RowKind binary(int nbytes) { return {true, nbytes}; }
    size_t row_bytes() const { return bin ? (size_t)dim : (size_t)dim * sizeof(float); }
    int check_dim(const char* who) const;                          // ERP_E_DIM outside the kind's range
    // engine of a search of nq rows against nt under ctx->engine: ERP_ENGINE_EXACT_SIMT, _TCGEN05 or _TCGEN05_1X.  Float
    // rows on a shape a forced tensor engine cannot serve: ERP_E_DIM, or SIMT with `fallback` (the cross-check search).
    int engine(erp_ctx* ctx, int nq, int nt, bool fallback, int* out) const;
    // the 2-NN on that engine.  `forward`: the search of the query rows; float rows record the SIMT search's statistics
    // and timing here (the other searches record their own), the cross-check search leaves them to the forward one.
    int knn2(erp_ctx* ctx, int engine, bool forward, const void* d_q, int nq, const void* d_t, int nt,
             int32_t* d_idx2, float* d_dist2, double* d_d2) const;
};
int check_knn_args(const char* who, erp_ctx* ctx, int nq, int nt, RowKind k);
int check_ransac_args(const char* who, erp_ctx* ctx, int H, int S, int metric, uint64_t hyp_offset);
// the keypoint, RANSAC and output arguments of a pair call (erp_pair_pose*), in the order of the C ABI: host pointers for
// a host-buffer call, device pointers for a device call
struct PairArgs {
    float ratio;
    int cross_check;
    const void *left_xy, *right_xy;
    size_t kp_stride;
    int width, height;
    uint64_t seed;
    int H, S, metric;
    float tau;
    erp_dmatch* matches;
    int32_t* n_matches;
    uint8_t* mask;
    erp_ransac_result* result;
};
// graph key of a device pair call: the entry's tag, then every argument.  It is compared bytewise: no padding bytes.
enum PairEntry : uint64_t { PAIR_F32 = 1, PAIR_BIN, PAIR_DIST };
struct PairKey {
    uint64_t entry;
    const void *q, *t;
    int64_t nq, nt, dim;
    PairArgs a;
};
static_assert(sizeof(PairArgs) == 8 * sizeof(uint64_t) + 8 * sizeof(int32_t) && sizeof(PairKey) == 6 * sizeof(uint64_t) + sizeof(PairArgs),
              "a pair-call graph key must have no padding bytes");
// graph cache (api.cu).  body: enqueues the call on ctx->stream without touching the host again.  The first call with a
// key runs directly, the second is captured, the rest replay.
int graph_run(erp_ctx* ctx, const PairKey& key, const std::function<int()>& body);
void graph_release(erp_ctx* ctx);
// host side of a pair call: waits for the stage event `ready` (the match list is final), brings back the matches (dev ->
// out) and the result; ERP_E_TOO_FEW_POINTS below S matches
int pair_pose_download(erp_ctx* ctx, const char* who, cudaEvent_t ready, const PairArgs& dev, const PairArgs& out);
int download_matches(erp_ctx* ctx, const erp_dmatch* d_out, const int32_t* d_n, size_t cap, erp_dmatch* out, int* n_out);
int upload_rows(erp_ctx* ctx, cudaStream_t stream, void* d_dst, const void* src, int rows, size_t row_bytes, size_t stride);
void stage_release(erp_ctx* ctx);
// multi-GPU (dist.cu)
int comm_allreduce_best(erp_ctx* ctx, uint64_t* d_packed);
void comm_release(erp_ctx* ctx);
int gather_bearings_chain(erp_ctx* ctx, const erp_dmatch* d_matches, int n_cap, const int32_t* d_n, const void* d_left_xy,
                          const void* d_right_xy, size_t stride, int q_offset, int W, int H, double* d_l3, double* d_r3,
                          float* d_l4, float* d_r4, float* Ks, int32_t* w);
int gather_slots_chain(erp_ctx* ctx, const erp_dmatch* d_slots, int n_ranks, int slot_records, int n_cap, erp_dmatch* d_out,
                       int32_t* d_n_out, const void* d_left_xy, const void* d_right_xy, size_t stride, int W, int H,
                       double* d_l3, double* d_r3, float* d_l4, float* d_r4, float* Ks, int32_t* w, uint32_t* ctl, const uint32_t* slot_flag);
int bearings_pair_chain(erp_ctx* ctx, const void* d_left_xy, const void* d_right_xy, size_t stride, int n, int W, int H,
                        double* d_l3, double* d_r3, float* d_l4, float* d_r4, float* Ks, int32_t* w);

} // namespace erp
