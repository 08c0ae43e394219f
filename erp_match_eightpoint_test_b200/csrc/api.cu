// api.cu -- context management, error reporting, host-pointer entry points (staging + copies)
// and the pieces of the reference's host logic that stay on the host (random_array replay).
#include "score_common.cuh"

#include <stdarg.h>

#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>

namespace erp {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

int Buf::reserve(size_t bytes)
{
    if (bytes <= cap) return ERP_OK;
    release();
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = host ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        p = nullptr; cap = 0;
        set_error("allocation of %zu bytes (%s) failed: %s", want, host ? "pinned" : "device", cudaGetErrorString(e));
        return ERP_E_CUDA;
    }
    cap = want;
    return ERP_OK;
}

void Buf::release()
{
    if (p) { if (host) cudaFreeHost(p); else cudaFree(p); }
    p = nullptr; cap = 0;
}

int gram_masked(erp_ctx*, const double*, const double*, int, const uint8_t*, double*);
int solve_batch(erp_ctx*, const double*, int, double*, float*, int max_sweeps = 30);
int consensus(erp_ctx*, const float*, int, float*, float*, int32_t*);
int mask_launch(erp_ctx*, const double*, const float*, const float*, int, int, float, uint8_t*, int32_t*);

// ---- host -> device of a (possibly strided) row matrix ------------------------------------------------------------
// Pinned sources go straight to the copy engine.  PAGEABLE sources -- what the C++ classes receive: a cv::Mat is plain
// heap memory -- are staged by a few host threads through pinned chunks: every thread copies its share of the rows
// into one of its two pinned slots (memcpy, ~10 GB/s per core) while the DMA of its other slot is in flight.  The
// driver's own pageable path is a single-threaded version of the same and was 2.2x slower for the 51 MB of cfg3.
constexpr size_t STAGE_CHUNK = 1 << 20;          // bytes per pinned slot
constexpr size_t STAGE_MIN_BYTES = 4 << 20;      // below this the driver's path is fine
// The helper threads live as long as the context: starting three threads per upload (and their first CUDA call) cost
// ~0.3 ms per call, more than the copy itself for one query chunk (scripts/stage_probe.py).
struct StagePool {
    static constexpr int THREADS = 8, SLOTS = 2;      // THREADS: upper bound; `threads` of them are used
    int threads = 4;                                  // $ERP_B200_STAGE_THREADS (1..8); thread 0 is the caller
    cudaStream_t stream[THREADS] = {};
    cudaEvent_t ev[THREADS][SLOTS] = {};
    uint8_t* pinned = nullptr;
    bool ok = false;
    // job hand-off: the caller publishes `job`, bumps `seq`; every helper runs job(t) once per seq
    std::thread helpers[THREADS - 1];
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    const std::function<void(int)>* job = nullptr;
    uint64_t seq = 0;
    int pending = 0;
    bool quit = false;

    void helper_main(int t, int device)
    {
        cudaSetDevice(device);
        uint64_t seen = 0;
        for (;;) {
            const std::function<void(int)>* j;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_job.wait(lk, [&] { return quit || seq != seen; });
                if (quit) return;
                seen = seq; j = job;
            }
            (*j)(t);
            {
                std::lock_guard<std::mutex> lk(mu);
                if (--pending == 0) cv_done.notify_one();
            }
        }
    }
    // runs work(t) for t = 0 .. threads-1 (0 on the calling thread) and returns when all are done
    void run(const std::function<void(int)>& work)
    {
        if (threads > 1) {
            std::lock_guard<std::mutex> lk(mu);
            job = &work; pending = threads - 1; seq++;
        }
        if (threads > 1) cv_job.notify_all();
        work(0);
        if (threads > 1) {
            std::unique_lock<std::mutex> lk(mu);
            cv_done.wait(lk, [&] { return pending == 0; });
            job = nullptr;
        }
    }
};

void stage_release(erp_ctx* ctx)
{
    StagePool* p = ctx->stage;
    if (!p) return;
    {
        std::lock_guard<std::mutex> lk(p->mu);
        p->quit = true;
    }
    p->cv_job.notify_all();
    for (auto& h : p->helpers) if (h.joinable()) h.join();
    for (int t = 0; t < StagePool::THREADS; t++) {
        if (p->stream[t]) { cudaStreamSynchronize(p->stream[t]); cudaStreamDestroy(p->stream[t]); }
        for (int s = 0; s < StagePool::SLOTS; s++) if (p->ev[t][s]) cudaEventDestroy(p->ev[t][s]);
    }
    if (p->pinned) cudaFreeHost(p->pinned);
    delete p;
    ctx->stage = nullptr;
}

static StagePool* stage_pool(erp_ctx* ctx)
{
    if (ctx->stage) return ctx->stage->ok ? ctx->stage : nullptr;
    StagePool* p = ctx->stage = new StagePool();
    if (const char* e = getenv("ERP_B200_STAGE_THREADS")) { const int n = atoi(e); if (n >= 1 && n <= StagePool::THREADS) p->threads = n; }
    bool ok = cudaMallocHost(&p->pinned, STAGE_CHUNK * StagePool::THREADS * StagePool::SLOTS) == cudaSuccess;
    for (int t = 0; t < p->threads && ok; t++) {
        ok = cudaStreamCreateWithFlags(&p->stream[t], cudaStreamNonBlocking) == cudaSuccess;
        for (int s = 0; s < StagePool::SLOTS && ok; s++) ok = cudaEventCreateWithFlags(&p->ev[t][s], cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) cudaGetLastError();
    if (ok) for (int t = 1; t < p->threads; t++) p->helpers[t - 1] = std::thread(&StagePool::helper_main, p, t, ctx->device);
    p->ok = ok;
    return ok ? p : nullptr;
}

static double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

static bool is_pageable(const void* p)
{
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return a.type == cudaMemoryTypeUnregistered;
}

int upload_rows(erp_ctx* ctx, cudaStream_t stream, void* d_dst, const void* src, int rows, size_t row_bytes, size_t stride)
{
    if (rows == 0) return ERP_OK;
    const size_t total = row_bytes * (size_t)rows;
    StagePool* pool = (total >= STAGE_MIN_BYTES && row_bytes <= STAGE_CHUNK && is_pageable(src)) ? stage_pool(ctx) : nullptr;
    if (!pool) {
        if (stride == row_bytes) ERP_CUDA(cudaMemcpyAsync(d_dst, src, total, cudaMemcpyHostToDevice, stream));
        else ERP_CUDA(cudaMemcpy2DAsync(d_dst, row_bytes, src, stride, row_bytes, rows, cudaMemcpyHostToDevice, stream));
        return ERP_OK;
    }
    // the staged copies must not overtake work already queued on the target buffer
    const double t_begin = now_s();
    ERP_CUDA(cudaEventRecord(ctx->ev_copy[8], stream));
    const int T = pool->threads;
    const int rows_per_chunk = (int)(STAGE_CHUNK / row_bytes);
    std::atomic<int> failed{0};
    const std::function<void(int)> work = [&](int t) {
        const int r0 = (int)((long long)rows * t / T), r1 = (int)((long long)rows * (t + 1) / T);
        if (cudaStreamWaitEvent(pool->stream[t], ctx->ev_copy[8], 0) != cudaSuccess) { failed = 1; return; }
        int slot = 0;
        for (int r = r0; r < r1; r += rows_per_chunk, slot ^= 1) {
            const int n = r1 - r < rows_per_chunk ? r1 - r : rows_per_chunk;
            uint8_t* buf = pool->pinned + ((size_t)t * StagePool::SLOTS + slot) * STAGE_CHUNK;
            if (cudaEventSynchronize(pool->ev[t][slot]) != cudaSuccess) { failed = 1; return; }       // the slot's previous DMA is done
            const uint8_t* s = static_cast<const uint8_t*>(src) + (size_t)r * stride;
            if (stride == row_bytes) memcpy(buf, s, (size_t)n * row_bytes);
            else for (int i = 0; i < n; i++) memcpy(buf + (size_t)i * row_bytes, s + (size_t)i * stride, row_bytes);
            if (cudaMemcpyAsync(static_cast<uint8_t*>(d_dst) + (size_t)r * row_bytes, buf, (size_t)n * row_bytes, cudaMemcpyHostToDevice,
                                pool->stream[t]) != cudaSuccess ||
                cudaEventRecord(pool->ev[t][slot], pool->stream[t]) != cudaSuccess) { failed = 1; return; }
        }
    };
    pool->run(work);
    if (failed) { set_error("staged upload failed: %s", cudaGetErrorString(cudaGetLastError())); return ERP_E_CUDA; }
    // `stream` continues after the last DMA of every helper stream
    for (int t = 0; t < T; t++)
        for (int s = 0; s < StagePool::SLOTS; s++) ERP_CUDA(cudaStreamWaitEvent(stream, pool->ev[t][s], 0));
    if (getenv("ERP_B200_STAGE_TRACE")) fprintf(stderr, "[stage] %zu bytes staged by %d threads, host %.3f ms\n", total, T, 1e3 * (now_s() - t_begin));
    return ERP_OK;
}

// Match records of a host-buffer call back to the caller in ONE round trip: the count and the record array (capacity
// `cap`) land in a pinned bounce buffer together, then the n records are copied out.  Waiting for the count first costs
// a second synchronisation, and a pageable `out` the driver's staged copy on top.
int download_matches(erp_ctx* ctx, const erp_dmatch* d_out, const int32_t* d_n, size_t cap, erp_dmatch* out, int* n_out)
{
    int32_t n = 0;
    int st = ERP_OK;
    const size_t cap_bytes = sizeof(erp_dmatch) * cap;
    if (cap_bytes <= (size_t)(8u << 20)) {
        uint8_t* h = ctx->host_scratch<uint8_t>(0, cap_bytes + 16, &st);
        ERP_TRY(st);
        ERP_CUDA(cudaMemcpyAsync(h, d_n, sizeof n, cudaMemcpyDeviceToHost, ctx->stream));
        if (cap_bytes) ERP_CUDA(cudaMemcpyAsync(h + 16, d_out, cap_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        ERP_CUDA(cudaStreamSynchronize(ctx->stream));
        memcpy(&n, h, sizeof n);
        if (n > 0) memcpy(out, h + 16, sizeof(erp_dmatch) * (size_t)n);
    } else {
        ERP_CUDA(cudaMemcpyAsync(&n, d_n, sizeof n, cudaMemcpyDeviceToHost, ctx->stream));
        ERP_CUDA(cudaStreamSynchronize(ctx->stream));
        if (n > 0) {
            ERP_CUDA(cudaMemcpyAsync(out, d_out, sizeof(erp_dmatch) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
            ERP_CUDA(cudaStreamSynchronize(ctx->stream));
        }
    }
    *n_out = n;
    return ERP_OK;
}

} // namespace erp

using namespace erp;

// ======================================================================================
ERP_API const char* erp_last_error(void) { return g_err; }
ERP_API int erp_version(void) { return ERP_B200_VERSION; }

ERP_API int erp_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

ERP_API int erp_ctx_create(int device, erp_ctx** out)
{
    ERP_ARG(out, ERP_E_ARG, "erp_ctx_create: out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        set_error("no CUDA device available (%s); this library has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
        return ERP_E_NO_DEVICE;
    }
    ERP_ARG(device >= 0 && device < n, ERP_E_ARG, "erp_ctx_create: device %d out of range [0,%d)", device, n);
    cudaDeviceProp prop;
    ERP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return ERP_E_ARCH;
    }
    DeviceGuard g(device);
    erp_ctx* ctx = new erp_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e));
        delete ctx;
        return ERP_E_CUDA;
    }
    bool ok = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreate(&ctx->ev_k0) == cudaSuccess && cudaEventCreate(&ctx->ev_k1) == cudaSuccess;
    for (auto& e2 : ctx->ev_stage) ok = ok && cudaEventCreate(&e2) == cudaSuccess;
    for (auto& e2 : ctx->ev_copy) ok = ok && cudaEventCreateWithFlags(&e2, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        set_error("cudaStreamCreate / cudaEventCreate failed");
        erp_ctx_destroy(ctx);
        return ERP_E_CUDA;
    }
    *out = ctx;
    return ERP_OK;
}

ERP_API void erp_ctx_destroy(erp_ctx* ctx)
{
    if (!ctx) return;
    DeviceGuard g(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    for (cudaEvent_t e : ctx->ev_copy) if (e) cudaEventDestroy(e);
    for (auto& b : ctx->dev) b.release();
    for (auto& b : ctx->pinned) b.release();
    if (ctx->ev_k0) cudaEventDestroy(ctx->ev_k0);
    if (ctx->ev_k1) cudaEventDestroy(ctx->ev_k1);
    for (cudaEvent_t e : ctx->ev_stage) if (e) cudaEventDestroy(e);
    comm_release(ctx);
    graph_release(ctx);
    stage_release(ctx);
    for (cudaEvent_t e : ctx->ev_score) cudaEventDestroy(e);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

ERP_API void* erp_ctx_stream(erp_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
ERP_API int erp_ctx_device(erp_ctx* ctx) { return ctx ? ctx->device : -1; }
ERP_API uint64_t erp_ctx_launch_count(erp_ctx* ctx) { return ctx ? ctx->launches : 0; }

ERP_API int erp_ctx_synchronize(erp_ctx* ctx)
{
    ERP_ARG(ctx, ERP_E_ARG, "null context");
    DeviceGuard g(ctx->device);
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

ERP_API int erp_ctx_set_engine(erp_ctx* ctx, int engine)
{
    ERP_ARG(ctx && engine >= ERP_ENGINE_AUTO && engine <= ERP_ENGINE_TCGEN05_1X, ERP_E_ARG, "erp_ctx_set_engine: bad argument");
    ctx->engine = engine;
    return ERP_OK;
}

ERP_API int erp_ctx_last_knn_kernel_ms(erp_ctx* ctx, float* ms)
{
    ERP_ARG(ctx && ms, ERP_E_ARG, "erp_ctx_last_knn_kernel_ms: bad argument");
    DeviceGuard g(ctx->device);
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    ERP_CUDA(cudaEventElapsedTime(ms, ctx->ev_k0, ctx->ev_k1));
    return ERP_OK;
}

ERP_API int erp_ctx_last_score_kernel_ms(erp_ctx* ctx, float* ms, int* launches)
{
    ERP_ARG(ctx && ms, ERP_E_ARG, "erp_ctx_last_score_kernel_ms: bad argument");
    DeviceGuard g(ctx->device);
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    float total = 0.f;
    for (int i = 0; i + 1 < ctx->n_ev_score; i += 2) {
        float t = 0.f;
        ERP_CUDA(cudaEventElapsedTime(&t, ctx->ev_score[i], ctx->ev_score[i + 1]));
        total += t;
    }
    *ms = total;
    if (launches) *launches = ctx->n_ev_score / 2;
    return ERP_OK;
}

ERP_API int erp_ctx_last_stage_ms(erp_ctx* ctx, float out[3])
{
    ERP_ARG(ctx && out, ERP_E_ARG, "erp_ctx_last_stage_ms: bad argument");
    DeviceGuard g(ctx->device);
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 3; i++) ERP_CUDA(cudaEventElapsedTime(&out[i], ctx->ev_stage[i], ctx->ev_stage[i + 1]));
    return ERP_OK;
}

ERP_API int erp_ctx_last_score_stats(erp_ctx* ctx, int64_t out[6])
{
    ERP_ARG(ctx && out, ERP_E_ARG, "erp_ctx_last_score_stats: bad argument");
    for (int i = 0; i < 6; i++) out[i] = 0;
    if (!ctx->sc_misc_dev) return ERP_OK;
    DeviceGuard g(ctx->device);
    int32_t w[W_WORDS];
    ERP_CUDA(cudaMemcpyAsync(w, ctx->sc_misc_dev, sizeof w, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    out[0] = w[W_DYN_A];       // hypotheses of the chunk
    out[1] = w[W_DYN_B + 2];   // correspondence tiles (of 256) every hypothesis was bounded on
    out[2] = w[W_NCT];         // correspondence tiles in total
    out[3] = w[W_DYN_C];       // survivors that were bounded on the rest
    out[4] = w[W_LENF];        // contenders scored exactly
    out[5] = w[W_LSTAR];       // L*: exact count of the first contender
    return ERP_OK;
}

ERP_API int erp_ctx_last_knn_stats(erp_ctx* ctx, int64_t out[5])
{
    ERP_ARG(ctx && out, ERP_E_ARG, "erp_ctx_last_knn_stats: bad argument");
    memcpy(out, ctx->knn_stats, sizeof ctx->knn_stats);
    if ((ctx->knn_stats[0] == ERP_ENGINE_TCGEN05 || ctx->knn_stats[0] == ERP_ENGINE_TCGEN05_1X) && ctx->tc_misc_dev) {
        // the re-scan count and the observed deviation live on the device
        DeviceGuard g(ctx->device);
        int32_t w[5] = {0, 0, 0, 0, 0};
        ERP_CUDA(cudaMemcpyAsync(w, ctx->tc_misc_dev, sizeof w, cudaMemcpyDeviceToHost, ctx->stream));
        ERP_CUDA(cudaStreamSynchronize(ctx->stream));
        out[1] = w[4];                              // summed over the query chunks of a host-buffer call
        float dev;
        memcpy(&dev, &w[2], 4);
        out[4] = (int64_t)((double)dev * 1e12);     // max |s_tc - s_exact| / (|q|^2 + max|t|^2), in 1e-12 units
    }
    return ERP_OK;
}

ERP_API int erp_ctx_last_knn_operands(erp_ctx* ctx, int64_t out[3])
{
    ERP_ARG(ctx && out, ERP_E_ARG, "erp_ctx_last_knn_operands: bad argument");
    const int64_t engine = ctx->knn_stats[0];
    out[0] = engine == ERP_ENGINE_TCGEN05 ? ERP_OPERANDS_TF32
           : engine == ERP_ENGINE_TCGEN05_1X ? (ctx->knn_bin ? ERP_OPERANDS_I8 : ERP_OPERANDS_F16)
           : ERP_OPERANDS_NONE;
    out[1] = out[2] = 0;
    if (out[0] == ERP_OPERANDS_F16 && ctx->tc_misc_dev) {
        DeviceGuard g(ctx->device);
        int32_t w[7] = {0, 0, 0, 0, 0, 0, 0};
        ERP_CUDA(cudaMemcpyAsync(w, ctx->tc_misc_dev, sizeof w, cudaMemcpyDeviceToHost, ctx->stream));
        ERP_CUDA(cudaStreamSynchronize(ctx->stream));
        out[1] = w[5] != 0;
        out[2] = w[6];
    }
    return ERP_OK;
}

// ======================================================================================
// matching: float rows (knn_exact.cu, knn_tc.cu, knn_tc1.cu) and binary rows (knn_bin.cu: feature_matcher::match_two_image
// with NORM_HAMMING) through the same entry points
// ======================================================================================
namespace erp {

int RowKind::check_dim(const char* who) const
{
    if (bin) ERP_ARG(dim >= 1 && dim <= 64, ERP_E_DIM, "%s: binary descriptor size %d must be in [1,64] bytes", who, dim);
    else ERP_ARG(dim > 0 && dim % 4 == 0 && dim <= 512, ERP_E_DIM, "%s: descriptor dimension %d must be a multiple of 4 in [4,512]", who, dim);
    return ERP_OK;
}

// Both tensor engine settings select the kind::i8 engine for binary rows, which serves every shape.  AUTO takes a tensor
// engine where it is faster than SIMT: the one-product engine for float rows, the i8 engine for binary rows.
int RowKind::engine(erp_ctx* ctx, int nq, int nt, bool fallback, int* out) const
{
    const bool forced = ctx->engine == ERP_ENGINE_TCGEN05 || ctx->engine == ERP_ENGINE_TCGEN05_1X;
    const bool tc = bin ? forced || (ctx->engine == ERP_ENGINE_AUTO && knn2_bin_preferred(nq, nt))
                        : forced ? knn2_tc_supported(nq, nt, dim) : ctx->engine == ERP_ENGINE_AUTO && knn2_tc_preferred(nq, nt, dim);
    ERP_ARG(tc || !forced || fallback, ERP_E_DIM, "tcgen05 engine does not support nq=%d nt=%d dim=%d", nq, nt, dim);
    *out = !tc ? ERP_ENGINE_EXACT_SIMT : ctx->engine == ERP_ENGINE_TCGEN05 ? ERP_ENGINE_TCGEN05 : ERP_ENGINE_TCGEN05_1X;
    return ERP_OK;
}

int RowKind::knn2(erp_ctx* ctx, int engine, bool forward, const void* d_q, int nq, const void* d_t, int nt,
                  int32_t* d_idx2, float* d_dist2, double* d_d2) const
{
    if (bin)
        return knn2_bin(ctx, static_cast<const uint8_t*>(d_q), nq, static_cast<const uint8_t*>(d_t), nt, dim, engine != ERP_ENGINE_EXACT_SIMT,
                        d_idx2, d_dist2, d_d2);
    const float *q = static_cast<const float*>(d_q), *t = static_cast<const float*>(d_t);
    if (engine == ERP_ENGINE_TCGEN05) return knn2_tc(ctx, q, nq, t, nt, dim, d_idx2, d_dist2, d_d2);
    if (engine == ERP_ENGINE_TCGEN05_1X) return knn2_tc1(ctx, q, nq, t, nt, dim, d_idx2, d_dist2, d_d2);
    if (!forward) return knn2_exact(ctx, q, nq, t, nt, dim, nullptr, 0, 0, d_idx2, d_dist2, d_d2);
    set_knn_stats(ctx, ERP_ENGINE_EXACT_SIMT, false, 1, cdiv(nq, 64), 0, nullptr);
    ERP_CUDA(record_timing(ctx, ctx->ev_k0));
    ERP_TRY(knn2_exact(ctx, q, nq, t, nt, dim, nullptr, 0, 0, d_idx2, d_dist2, d_d2));
    ERP_CUDA(record_timing(ctx, ctx->ev_k1));
    return ERP_OK;
}

int check_knn_args(const char* who, erp_ctx* ctx, int nq, int nt, RowKind k)
{
    ERP_ARG(ctx, ERP_E_ARG, "%s: null context", who);
    ERP_ARG(nq >= 0 && nt >= 0, ERP_E_ARG, "%s: negative size", who);
    ERP_TRY(k.check_dim(who));
    // knnMatch(k=2) on fewer than 2 train rows throws in the reference (FLANN: knn <= index size)
    ERP_ARG(nq == 0 || nt >= 2, ERP_E_TOO_FEW_TRAIN, "%s: k=2 needs at least 2 train descriptors, got %d", who, nt);
    return ERP_OK;
}

__global__ void add_offset_kernel(int32_t* v, int n, int off)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && v[i] >= 0) v[i] += off;
}

} // namespace erp

static int knn2_dev(const char* who, erp_ctx* ctx, RowKind k, const void* d_q, int nq, const void* d_t, int nt,
                    int32_t* d_idx2, float* d_dist2, double* d_d2)
{
    ERP_TRY(check_knn_args(who, ctx, nq, nt, k));
    if (nq == 0) return ERP_OK;
    ERP_ARG(d_q && d_t, ERP_E_ARG, "%s: null descriptors", who);
    DeviceGuard g(ctx->device);
    int engine;
    ERP_TRY(k.engine(ctx, nq, nt, false, &engine));
    return k.knn2(ctx, engine, true, d_q, nq, d_t, nt, d_idx2, d_dist2, d_d2);
}

// cross-check: the nearest query of every train row (roles swapped, lowest query index on ties), compacted to the first
// neighbour; the query index is offset by q_offset, d_best_d2 (float rows) receives the squared distance
static int knn1_reverse(erp_ctx* ctx, RowKind k, const void* d_q, int nq, const void* d_t, int nt, int q_offset,
                        int32_t* d_best_q, double* d_best_d2)
{
    int st = ERP_OK;
    int32_t* idx2 = ctx->scratch<int32_t>(S_RS_IDX, (size_t)nt * 2, &st);
    double* d2 = k.bin ? nullptr : ctx->scratch<double>(S_RS_D2, (size_t)nt * 2, &st);
    ERP_TRY(st);
    int engine;
    ERP_TRY(k.engine(ctx, nt, nq, true, &engine));
    ERP_TRY(k.knn2(ctx, engine, false, d_t, nt, d_q, nq, idx2, nullptr, d2));      // (no index offset: it is added below)
    ERP_CUDA(cudaMemcpy2DAsync(d_best_q, sizeof(int32_t), idx2, 2 * sizeof(int32_t), sizeof(int32_t), nt,
                               cudaMemcpyDeviceToDevice, ctx->stream));
    if (d_best_d2)
        ERP_CUDA(cudaMemcpy2DAsync(d_best_d2, sizeof(double), d2, 2 * sizeof(double), sizeof(double), nt,
                                   cudaMemcpyDeviceToDevice, ctx->stream));
    if (q_offset != 0) {
        erp::add_offset_kernel<<<cdiv(nt, 256), 256, 0, ctx->stream>>>(d_best_q, nt, q_offset);
        ERP_LAUNCH(ctx, "add_offset_kernel");
    }
    return ERP_OK;
}

// the cross-check (when asked) and the ratio filter of the 2-NN of a pair: match records and their count on the device
static int filter_matches(erp_ctx* ctx, RowKind k, const void* d_q, int nq, const void* d_t, int nt, const int32_t* idx2,
                          const float* dist2, float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out)
{
    int32_t* rev = nullptr;
    if (cross_check && nq > 0) {
        int st = ERP_OK;
        rev = ctx->scratch<int32_t>(S_REVQ, (size_t)nt, &st);
        ERP_TRY(st);
        ERP_TRY(knn1_reverse(ctx, k, d_q, nq, d_t, nt, 0, rev, nullptr));
    }
    return erp_match_filter_dev(ctx, idx2, dist2, nq, ratio, rev, 0, d_out, d_n_out);
}

static int knn2_match_dev(const char* who, erp_ctx* ctx, RowKind k, const void* d_q, int nq, const void* d_t, int nt,
                          float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out)
{
    ERP_TRY(check_knn_args(who, ctx, nq, nt, k));
    ERP_ARG(d_n_out, ERP_E_ARG, "%s: d_n_out is null", who);
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    int32_t* idx2 = ctx->scratch<int32_t>(S_IDX2, (size_t)nq * 2 + 2, &st);
    float* dist2 = ctx->scratch<float>(S_DIST2, (size_t)nq * 2 + 2, &st);
    ERP_TRY(st);
    ERP_TRY(knn2_dev(who, ctx, k, d_q, nq, d_t, nt, idx2, dist2, nullptr));
    return filter_matches(ctx, k, d_q, nq, d_t, nt, idx2, dist2, ratio, cross_check, d_out, d_n_out);
}

// Host-buffer 2-NN: the train set and the first query chunk are uploaded, then every further query chunk travels
// (on its own stream) while the previous one is searched.  Rows are independent, so the result does not depend on
// the cut; the train-side operands are prepared by the first chunk only.
//
// The cut (scripts/stage_probe.py prints the device timeline of a call; cfg3, 100k x 100k x 64): a chunk's search costs
// ~0.10 ms + 17.5 us per 1000 rows, the train set must be complete before anything starts (0.47 ms pinned, ~1 ms staged
// from pageable memory), and after the first chunk the call is search bound.  So the FIRST chunk is short -- it only has
// to cover the upload of the second -- and the number of chunks small: two from pinned memory (5/32 + 27/32), three from
// pageable memory where the staging is slower than the search (1/8 + 3/8 + 1/2).  $ERP_B200_HOST_CHUNKS = 1..7 forces a
// count (a short first chunk, then even ones).  Small inputs: one chunk.
static int chunk_bounds(int nq, int nt, bool pageable, int (&bounds)[9])
{
    static int forced = -1;
    if (forced < 0) {
        const char* e = getenv("ERP_B200_HOST_CHUNKS");
        forced = e ? atoi(e) : 0;
        if (forced < 0 || forced > 7) forced = 0;
    }
    auto round256 = [](long long v) { return (int)((v + 255) / 256 * 256); };
    int n = 0;
    bounds[0] = 0;
    auto cut = [&](int r) { if (r > bounds[n] && r < nq) bounds[++n] = r; };
    if (forced > 1) {
        const int first = forced > 2 ? round256(cdiv(nq, 2 * forced)) : 0;
        cut(first);
        const int rows = round256(cdiv(nq - bounds[n], forced - n));
        for (int r = bounds[n] + rows; r < nq; r += rows) cut(r);
    } else if (forced == 0 && (double)nq * (double)nt >= 4.0e9) {
        if (pageable) { cut(round256(nq / 8)); cut(round256(nq / 2)); }
        else cut(round256((long long)nq * 5 / 32));
    }
    bounds[++n] = nq;
    return n;
}

// host rows -> S_Q / S_T (dense, 16 bytes of padding) and their 2-NN
static int knn2_host(erp_ctx* ctx, RowKind k, const void* q, int nq, size_t qs, const void* t, int nt, size_t ts,
                     int32_t* d_idx2, float* d_dist2)
{
    const size_t row = k.row_bytes();
    ERP_ARG((nq == 0 || q) && (nt == 0 || t), ERP_E_ARG, "null descriptor pointer");
    ERP_ARG(qs >= row && ts >= row, ERP_E_ARG, "row stride smaller than a descriptor row (%zu < %zu)", qs < ts ? qs : ts, row);
    int st = ERP_OK;
    uint8_t* dq = ctx->scratch<uint8_t>(S_Q, (size_t)nq * row + 16, &st);
    uint8_t* dt = ctx->scratch<uint8_t>(S_T, (size_t)nt * row + 16, &st);
    ERP_TRY(st);
    // one engine for the whole call: the tensor engines prepare the train operand with the first query chunk only
    int engine;
    ERP_TRY(k.engine(ctx, nq, nt, false, &engine));
    int bounds[9];
    const int chunks = chunk_bounds(nq, nt, is_pageable(q), bounds);
    // fork: the copy stream starts after whatever the context stream still has queued
    ERP_CUDA(cudaEventRecord(ctx->ev_copy[7], ctx->stream));
    ERP_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy[7], 0));
    // tc_chunk > 0 tells the tensor engines that the train operand of this call is already prepared: it must not
    // survive this function on ANY exit path (a stale value would make the next call reuse old train data)
    struct ChunkReset { erp_ctx* c; ~ChunkReset() { c->tc_chunk = 0; } } reset{ctx};
    // $ERP_B200_STAGE_TRACE: device-side timeline of the call (uploads on the copy stream, searches on the context stream)
    const bool trace = getenv("ERP_B200_STAGE_TRACE") != nullptr;
    cudaEvent_t tr[20] = {};
    int n_tr = 0;
    auto mark = [&](cudaStream_t s) { if (trace && n_tr < 20 && cudaEventCreate(&tr[n_tr]) == cudaSuccess) cudaEventRecord(tr[n_tr++], s); };
    mark(ctx->copy_stream);
    int rc = upload_rows(ctx, ctx->copy_stream, dt, t, nt, row, ts);
    mark(ctx->copy_stream);
    // chunk c's search is enqueued as soon as chunk c is on its way: a pageable source blocks this thread while the
    // staging threads copy chunk c + 1, and the device searches chunk c meanwhile (pinned sources never block here)
    for (int c = 0; c < chunks && rc == ERP_OK; c++) {
        const int r0 = bounds[c], n = bounds[c + 1] - r0;
        rc = upload_rows(ctx, ctx->copy_stream, dq + (size_t)r0 * row, static_cast<const char*>(q) + (size_t)r0 * qs, n, row, qs);
        if (rc == ERP_OK && cudaEventRecord(ctx->ev_copy[c], ctx->copy_stream) != cudaSuccess) rc = ERP_E_CUDA;
        mark(ctx->copy_stream);
        if (rc != ERP_OK) break;
        ERP_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy[c], 0));
        mark(ctx->stream);
        ctx->tc_chunk = c;
        const double t_enq = now_s();
        rc = k.knn2(ctx, engine, true, dq + (size_t)r0 * row, n, dt, nt, d_idx2 + 2 * (size_t)r0, d_dist2 + 2 * (size_t)r0, nullptr);
        mark(ctx->stream);
        if (trace) fprintf(stderr, "[stage] chunk %d: search of %d rows enqueued in %.3f ms (host)\n", c, n, 1e3 * (now_s() - t_enq));
    }
    if (trace && n_tr > 0) {
        // marks: 0 fork, 1 train up, then per chunk { upload done (copy stream), search start, search end (context stream) }
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->copy_stream);
        fprintf(stderr, "[stage] device timeline (ms after the fork):");
        for (int i = 1; i < n_tr; i++) { float ms = 0.f; cudaEventElapsedTime(&ms, tr[0], tr[i]); fprintf(stderr, " %.3f", ms); }
        fprintf(stderr, "\n");
        for (int i = 0; i < n_tr; i++) cudaEventDestroy(tr[i]);
    }
    return rc;
}

static int knn2_match_host(const char* who, erp_ctx* ctx, RowKind k, const void* q, int nq, size_t qs, const void* t, int nt,
                           size_t ts, float ratio, int cross_check, erp_dmatch* out, int* n_out)
{
    ERP_TRY(check_knn_args(who, ctx, nq, nt, k));
    ERP_ARG(n_out, ERP_E_ARG, "%s: n_out is null", who);
    *n_out = 0;
    if (nq == 0) return ERP_OK;
    ERP_ARG(out, ERP_E_ARG, "%s: out is null", who);
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    erp_dmatch* d_out = ctx->scratch<erp_dmatch>(S_OUT, (size_t)nq, &st);
    int32_t* d_n = ctx->scratch<int32_t>(S_NOUT, 4, &st);
    int32_t* idx2 = ctx->scratch<int32_t>(S_IDX2, (size_t)nq * 2 + 2, &st);
    float* dist2 = ctx->scratch<float>(S_DIST2, (size_t)nq * 2 + 2, &st);
    ERP_TRY(st);
    ERP_TRY(knn2_host(ctx, k, q, nq, qs, t, nt, ts, idx2, dist2));
    ERP_TRY(filter_matches(ctx, k, ctx->dev[S_Q].p, nq, ctx->dev[S_T].p, nt, idx2, dist2, ratio, cross_check, d_out, d_n));
    return download_matches(ctx, d_out, d_n, (size_t)nq, out, n_out);
}

static int knn2_raw_host(const char* who, erp_ctx* ctx, RowKind k, const void* q, int nq, size_t qs, const void* t, int nt,
                         size_t ts, int32_t* idx2, float* dist2)
{
    ERP_TRY(check_knn_args(who, ctx, nq, nt, k));
    if (nq == 0) return ERP_OK;
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    int32_t* d_idx = ctx->scratch<int32_t>(S_IDX2, (size_t)nq * 2 + 2, &st);
    float* d_dist = ctx->scratch<float>(S_DIST2, (size_t)nq * 2 + 2, &st);
    ERP_TRY(st);
    ERP_TRY(knn2_host(ctx, k, q, nq, qs, t, nt, ts, d_idx, d_dist));
    if (idx2) ERP_CUDA(cudaMemcpyAsync(idx2, d_idx, sizeof(int32_t) * 2 * (size_t)nq, cudaMemcpyDeviceToHost, ctx->stream));
    if (dist2) ERP_CUDA(cudaMemcpyAsync(dist2, d_dist, sizeof(float) * 2 * (size_t)nq, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

ERP_API int erp_knn2_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                         int32_t* d_idx2, float* d_dist2, double* d_d2)
{
    return knn2_dev("erp_knn2_dev", ctx, RowKind::f32(dim), d_q, nq, d_t, nt, d_idx2, d_dist2, d_d2);
}

ERP_API int erp_nn1_reverse_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                                int q_offset, int32_t* d_best_q, double* d_best_d2)
{
    ERP_ARG(ctx && nq >= 1 && nt >= 0 && d_best_q, ERP_E_ARG, "erp_nn1_reverse_dev: bad argument");
    ERP_TRY(RowKind::f32(dim).check_dim("erp_nn1_reverse_dev"));
    if (nt == 0) return ERP_OK;
    DeviceGuard g(ctx->device);
    return knn1_reverse(ctx, RowKind::f32(dim), d_q, nq, d_t, nt, q_offset, d_best_q, d_best_d2);
}

ERP_API int erp_knn2_match_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                               float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out)
{
    return knn2_match_dev("erp_knn2_match_dev", ctx, RowKind::f32(dim), d_q, nq, d_t, nt, ratio, cross_check, d_out, d_n_out);
}

ERP_API int erp_knn2_match(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes,
                           const float* t, int nt, size_t t_stride_bytes, int dim,
                           float ratio, int cross_check, erp_dmatch* out, int* n_out)
{
    return knn2_match_host("erp_knn2_match", ctx, RowKind::f32(dim), q, nq, q_stride_bytes, t, nt, t_stride_bytes, ratio, cross_check,
                           out, n_out);
}

ERP_API int erp_knn2_raw(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes,
                         const float* t, int nt, size_t t_stride_bytes, int dim,
                         int32_t* idx2, float* dist2)
{
    return knn2_raw_host("erp_knn2_raw", ctx, RowKind::f32(dim), q, nq, q_stride_bytes, t, nt, t_stride_bytes, idx2, dist2);
}

ERP_API int erp_knn2_near_ties(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes,
                               const float* t, int nt, size_t t_stride_bytes, int dim, float rel_tol,
                               uint8_t* flags, int* n_flagged)
{
    ERP_TRY(check_knn_args("erp_knn2_near_ties", ctx, nq, nt, RowKind::f32(dim)));
    ERP_ARG(n_flagged && rel_tol >= 0.f, ERP_E_ARG, "erp_knn2_near_ties: bad argument");
    *n_flagged = 0;
    if (nq == 0) return ERP_OK;
    ERP_ARG(flags, ERP_E_ARG, "erp_knn2_near_ties: flags is null");
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    int32_t* d_idx = ctx->scratch<int32_t>(S_IDX2, (size_t)nq * 2 + 2, &st);
    float* d_dist = ctx->scratch<float>(S_DIST2, (size_t)nq * 2 + 2, &st);
    double* d_d2 = ctx->scratch<double>(S_D2, (size_t)nq * 2 + 2, &st);
    int32_t* d_third = ctx->scratch<int32_t>(S_COUNTS, (size_t)nq + 1, &st);
    uint8_t* d_flags = ctx->scratch<uint8_t>(S_MASK, (size_t)nq + 4, &st);
    ERP_TRY(st);
    // the engine's own exact 2-NN (indices + fp64 squared distances), then one exact counting pass
    size_t row = (size_t)dim * sizeof(float);
    ERP_ARG(q && t && q_stride_bytes >= row && t_stride_bytes >= row, ERP_E_ARG, "erp_knn2_near_ties: bad descriptor buffers");
    float* dq = ctx->scratch<float>(S_Q, (size_t)nq * dim + 4, &st);
    float* dt = ctx->scratch<float>(S_T, (size_t)nt * dim + 4, &st);
    ERP_TRY(st);
    ERP_TRY(upload_rows(ctx, ctx->stream, dt, t, nt, row, t_stride_bytes));
    ERP_TRY(upload_rows(ctx, ctx->stream, dq, q, nq, row, q_stride_bytes));
    ERP_TRY(erp_knn2_dev(ctx, dq, nq, dt, nt, dim, d_idx, d_dist, d_d2));
    ERP_TRY(near_ties(ctx, dq, nq, dt, nt, dim, d_idx, d_d2, (double)rel_tol, d_third, d_flags));
    int32_t n = 0;
    ERP_CUDA(cudaMemcpyAsync(flags, d_flags, (size_t)nq, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaMemcpyAsync(&n, d_third + nq, sizeof n, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    *n_flagged = n;
    return ERP_OK;
}

ERP_API int erp_knn2_bin_dev(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes,
                             int32_t* d_idx2, float* d_dist2, double* d_d2)
{
    return knn2_dev("erp_knn2_bin_dev", ctx, RowKind::binary(nbytes), d_q, nq, d_t, nt, d_idx2, d_dist2, d_d2);
}

ERP_API int erp_knn2_match_bin_dev(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes,
                                   float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out)
{
    return knn2_match_dev("erp_knn2_match_bin_dev", ctx, RowKind::binary(nbytes), d_q, nq, d_t, nt, ratio, cross_check, d_out, d_n_out);
}

ERP_API int erp_knn2_match_bin(erp_ctx* ctx, const uint8_t* q, int nq, size_t q_stride_bytes,
                               const uint8_t* t, int nt, size_t t_stride_bytes, int nbytes,
                               float ratio, int cross_check, erp_dmatch* out, int* n_out)
{
    return knn2_match_host("erp_knn2_match_bin", ctx, RowKind::binary(nbytes), q, nq, q_stride_bytes, t, nt, t_stride_bytes, ratio,
                           cross_check, out, n_out);
}

ERP_API int erp_knn2_raw_bin(erp_ctx* ctx, const uint8_t* q, int nq, size_t q_stride_bytes,
                             const uint8_t* t, int nt, size_t t_stride_bytes, int nbytes,
                             int32_t* idx2, float* dist2)
{
    return knn2_raw_host("erp_knn2_raw_bin", ctx, RowKind::binary(nbytes), q, nq, q_stride_bytes, t, nt, t_stride_bytes, idx2, dist2);
}

// ======================================================================================
// geometry, host-pointer forms
// ======================================================================================
ERP_API int erp_bearings_from_pixels(erp_ctx* ctx, const void* xy, size_t stride_bytes, int n,
                                     int width, int height, double* out3)
{
    ERP_ARG(ctx && n >= 0 && width > 0 && height > 0, ERP_E_ARG, "erp_bearings_from_pixels: bad argument");
    ERP_ARG(stride_bytes >= 8 && stride_bytes % 4 == 0, ERP_E_ARG, "erp_bearings_from_pixels: bad stride %zu", stride_bytes);
    if (n == 0) return ERP_OK;
    ERP_ARG(xy && out3, ERP_E_ARG, "erp_bearings_from_pixels: null buffer");
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    float* d_xy = ctx->scratch<float>(S_XY, (size_t)n * 2, &st);
    double* d_o = ctx->scratch<double>(S_L3, (size_t)n * 3, &st);
    ERP_TRY(st);
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy, xy, n, 8, stride_bytes));
    ERP_TRY(erp_bearings_dev(ctx, d_xy, 8, n, width, height, d_o, nullptr));
    ERP_CUDA(cudaMemcpyAsync(out3, d_o, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

// upload m x 3 fp64 bearings for both views; optionally build the float4 copies
static int stage_bearings(erp_ctx* ctx, const double* l3, const double* r3, int m,
                          double** dl, double** dr, float** dl4, float** dr4)
{
    ERP_ARG(m == 0 || (l3 && r3), ERP_E_ARG, "null bearing pointer");
    int st = ERP_OK;
    *dl = ctx->scratch<double>(S_L3, (size_t)m * 3 + 4, &st);
    *dr = ctx->scratch<double>(S_R3, (size_t)m * 3 + 4, &st);
    ERP_TRY(st);
    if (m) {
        ERP_CUDA(cudaMemcpyAsync(*dl, l3, sizeof(double) * 3 * (size_t)m, cudaMemcpyHostToDevice, ctx->stream));
        ERP_CUDA(cudaMemcpyAsync(*dr, r3, sizeof(double) * 3 * (size_t)m, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (dl4) {
        *dl4 = ctx->scratch<float>(S_L4, (size_t)m * 4 + 4, &st);
        *dr4 = ctx->scratch<float>(S_R4, (size_t)m * 4 + 4, &st);
        ERP_TRY(st);
        ERP_TRY(erp_pack_float4_dev(ctx, *dl, m, *dl4));
        ERP_TRY(erp_pack_float4_dev(ctx, *dr, m, *dr4));
    }
    return ERP_OK;
}

ERP_API int erp_eight_point_batch(erp_ctx* ctx, const double* l3, const double* r3, int m,
                                  const int32_t* samples, int H, int S, uint64_t seed, uint64_t hyp_offset,
                                  double* E_out, float* pose_out)
{
    ERP_ARG(ctx && E_out && H >= 0 && m >= 0, ERP_E_ARG, "erp_eight_point_batch: bad argument");
    ERP_ARG(S >= 8 && m >= S, ERP_E_TOO_FEW_POINTS, "erp_eight_point_batch: sample size %d of %d correspondences (need 8 <= S <= m)", S, m);
    if (H == 0) return ERP_OK;
    DeviceGuard g(ctx->device);
    double *dl, *dr;
    ERP_TRY(stage_bearings(ctx, l3, r3, m, &dl, &dr, nullptr, nullptr));
    int st = ERP_OK;
    int32_t* d_s = nullptr;
    if (samples) {
        for (size_t i = 0; i < (size_t)H * S; i++)
            ERP_ARG(samples[i] >= 0 && samples[i] < m, ERP_E_ARG, "sample index %d out of range [0,%d)", samples[i], m);
        d_s = ctx->scratch<int32_t>(S_SAMPLES, (size_t)H * S, &st);
        ERP_TRY(st);
        ERP_CUDA(cudaMemcpyAsync(d_s, samples, sizeof(int32_t) * (size_t)H * S, cudaMemcpyHostToDevice, ctx->stream));
    }
    double* dE = ctx->scratch<double>(S_E, (size_t)H * 9, &st);
    float* dP = pose_out ? ctx->scratch<float>(S_POSE, (size_t)H * ERP_POSE_FLOATS, &st) : nullptr;
    ERP_TRY(st);
    ERP_TRY(erp_eight_point_batch_dev(ctx, dl, dr, m, d_s, H, S, seed, hyp_offset, dE, dP));
    ERP_CUDA(cudaMemcpyAsync(E_out, dE, sizeof(double) * 9 * (size_t)H, cudaMemcpyDeviceToHost, ctx->stream));
    if (pose_out) ERP_CUDA(cudaMemcpyAsync(pose_out, dP, sizeof(float) * ERP_POSE_FLOATS * (size_t)H, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

ERP_API int erp_refit(erp_ctx* ctx, const double* l3, const double* r3, int m, const uint8_t* mask,
                      double* E_out, float* pose_out)
{
    ERP_ARG(ctx && m >= 0 && (E_out || pose_out), ERP_E_ARG, "erp_refit: bad argument");
    int used = m;
    if (mask) { used = 0; for (int i = 0; i < m; i++) used += mask[i] != 0; }
    ERP_ARG(used >= 8, ERP_E_TOO_FEW_POINTS, "erp_refit: %d correspondences selected, need >= 8", used);
    DeviceGuard g(ctx->device);
    double *dl, *dr;
    ERP_TRY(stage_bearings(ctx, l3, r3, m, &dl, &dr, nullptr, nullptr));
    int st = ERP_OK;
    uint8_t* d_mask = nullptr;
    if (mask) {
        d_mask = ctx->scratch<uint8_t>(S_MASK, (size_t)m, &st);
        ERP_TRY(st);
        ERP_CUDA(cudaMemcpyAsync(d_mask, mask, (size_t)m, cudaMemcpyHostToDevice, ctx->stream));
    }
    double* misc = ctx->scratch<double>(S_MISC, 128, &st);
    ERP_TRY(st);
    double *G = misc, *E = misc + 45;
    float* pose = reinterpret_cast<float*>(misc + 54);
    ERP_TRY(gram_masked(ctx, dl, dr, m, d_mask, G));
    ERP_TRY(solve_batch(ctx, G, 1, E, pose));
    if (E_out) ERP_CUDA(cudaMemcpyAsync(E_out, E, sizeof(double) * 9, cudaMemcpyDeviceToHost, ctx->stream));
    if (pose_out) ERP_CUDA(cudaMemcpyAsync(pose_out, pose, sizeof(float) * ERP_POSE_FLOATS, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

// eight_point::eight_point_estimation(w, h, left, right, R1, R2, T, v1, v2, n)
ERP_API int erp_eight_point_estimation(erp_ctx* ctx, const double* l3, const double* r3, int n,
                                       double* E_out, float* R1_vec, float* R2_vec, float* T_vec,
                                       int* R1_valid, int* R2_valid)
{
    ERP_ARG(n >= 8, ERP_E_TOO_FEW_POINTS, "eight_point_estimation needs >= 8 correspondences, got %d", n);
    double E[9];
    float pose[ERP_POSE_FLOATS];
    ERP_TRY(erp_refit(ctx, l3, r3, n, nullptr, E, pose));
    if (E_out) memcpy(E_out, E, sizeof E);
    if (R1_vec) memcpy(R1_vec, pose, 12);
    if (R2_vec) memcpy(R2_vec, pose + 3, 12);
    if (T_vec) memcpy(T_vec, pose + 6, 12);
    if (R1_valid) *R1_valid = pose[9] != 0.f;
    if (R2_valid) *R2_valid = pose[10] != 0.f;
    return ERP_OK;
}

ERP_API int erp_score(erp_ctx* ctx, const double* E, int H, const double* l3, const double* r3, int m,
                      int metric, float tau, int32_t* counts)
{
    ERP_ARG(ctx && H >= 0 && m >= 0, ERP_E_ARG, "erp_score: bad argument");
    if (H == 0) return ERP_OK;
    ERP_ARG(E && counts, ERP_E_ARG, "erp_score: null buffer");
    DeviceGuard g(ctx->device);
    double *dl, *dr;
    float *dl4, *dr4;
    ERP_TRY(stage_bearings(ctx, l3, r3, m, &dl, &dr, &dl4, &dr4));
    int st = ERP_OK;
    double* dE = ctx->scratch<double>(S_E, (size_t)H * 9, &st);
    int32_t* dc = ctx->scratch<int32_t>(S_COUNTS, (size_t)H, &st);
    ERP_TRY(st);
    ERP_CUDA(cudaMemcpyAsync(dE, E, sizeof(double) * 9 * (size_t)H, cudaMemcpyHostToDevice, ctx->stream));
    ERP_TRY(erp_score_dev(ctx, dE, H, dl4, dr4, m, metric, tau, 0, dc, nullptr));
    ERP_CUDA(cudaMemcpyAsync(counts, dc, sizeof(int32_t) * (size_t)H, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

ERP_API int erp_inlier_mask(erp_ctx* ctx, const double* E9, const double* l3, const double* r3, int m,
                            int metric, float tau, uint8_t* mask, int* n_inliers)
{
    ERP_ARG(ctx && E9 && m >= 0, ERP_E_ARG, "erp_inlier_mask: bad argument");
    ERP_ARG(metric >= 0 && metric <= 2, ERP_E_ARG, "erp_inlier_mask: unknown metric %d", metric);
    DeviceGuard g(ctx->device);
    double *dl, *dr;
    float *dl4, *dr4;
    ERP_TRY(stage_bearings(ctx, l3, r3, m, &dl, &dr, &dl4, &dr4));
    int st = ERP_OK;
    double* misc = ctx->scratch<double>(S_MISC, 128, &st);
    uint8_t* d_mask = ctx->scratch<uint8_t>(S_MASK, (size_t)m + 4, &st);
    ERP_TRY(st);
    int32_t* d_n = reinterpret_cast<int32_t*>(misc + 16);
    ERP_CUDA(cudaMemcpyAsync(misc, E9, sizeof(double) * 9, cudaMemcpyHostToDevice, ctx->stream));
    ERP_TRY(mask_launch(ctx, misc, dl4, dr4, m, metric, tau, d_mask, d_n));
    int32_t n = 0;
    if (mask && m) ERP_CUDA(cudaMemcpyAsync(mask, d_mask, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaMemcpyAsync(&n, d_n, sizeof n, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n_inliers) *n_inliers = n;
    return ERP_OK;
}

namespace erp {

// ---- CUDA graph of a device-resident pair call ------------------------------------------------------------------
// One pair is ~25 stream operations of which most are a few microseconds long: issued one by one the host cannot stay
// ahead of the GPU (and, multi-GPU, the ranks drift apart between two collectives).  The calls that only enqueue
// (erp_pair_pose_dev, erp_pair_pose_dist_dev) are therefore captured: first call with a given argument set runs
// directly (it also sizes the scratch), the second one is captured into a graph, later ones are one cudaGraphLaunch.
// A cached graph holds device pointers: any scratch re-allocation, engine change or new clique invalidates it.
// ERP_B200_GRAPH=0 turns the cache off.
struct GraphCache {
    std::vector<uint8_t> key, seen;
    uint64_t key_gen = 0, seen_gen = 0;
    cudaGraphExec_t exec = nullptr;
    uint64_t launches = 0;
    int64_t knn_stats[5] = {0, 0, 0, 0, 0};
    bool knn_bin = false;
    int32_t *sc_misc_dev = nullptr, *tc_misc_dev = nullptr;
    int n_ev_score = 0;
    bool disabled = false;
};

void graph_release(erp_ctx* ctx)
{
    if (!ctx->graph) return;
    if (ctx->graph->exec) cudaGraphExecDestroy(ctx->graph->exec);
    delete ctx->graph;
    ctx->graph = nullptr;
}

int graph_run(erp_ctx* ctx, const PairKey& key, const std::function<int()>& body)
{
    static const bool off = [] { const char* e = getenv("ERP_B200_GRAPH"); return e && atoi(e) == 0; }();
    if (off) return body();
    if (!ctx->graph) ctx->graph = new GraphCache();
    GraphCache& g = *ctx->graph;
    if (g.disabled) return body();
    std::vector<uint8_t> k((const uint8_t*)&key, (const uint8_t*)&key + sizeof key);
    const void* extra[2] = {(const void*)(intptr_t)ctx->engine, (const void*)ctx->comm};
    k.insert(k.end(), (const uint8_t*)extra, (const uint8_t*)extra + sizeof extra);
    if (g.exec && g.key == k && g.key_gen == ctx->scratch_gen) {
        ERP_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
        ctx->launches += g.launches;
        memcpy(ctx->knn_stats, g.knn_stats, sizeof g.knn_stats);
        ctx->knn_bin = g.knn_bin;
        ctx->sc_misc_dev = g.sc_misc_dev; ctx->tc_misc_dev = g.tc_misc_dev; ctx->n_ev_score = g.n_ev_score;
        return ERP_OK;
    }
    if (g.seen == k && g.seen_gen == ctx->scratch_gen) {
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
        const uint64_t l0 = ctx->launches;
        if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
            cudaGetLastError();
            g.disabled = true;
            return body();
        }
        ctx->capturing = true;
        const int st = body();
        ctx->capturing = false;
        cudaGraph_t graph = nullptr;
        const cudaError_t e = cudaStreamEndCapture(ctx->stream, &graph);
        const bool usable = st == ERP_OK && e == cudaSuccess && graph && ctx->scratch_gen == g.seen_gen;
        if (usable && cudaGraphInstantiate(&g.exec, graph, 0) != cudaSuccess) g.exec = nullptr;
        if (graph) cudaGraphDestroy(graph);
        if (!usable || !g.exec) {
            // nothing was executed: run the call directly; a body that cannot be captured stays on the direct path
            cudaGetLastError();
            ctx->launches = l0;
            g.exec = nullptr;
            g.seen.clear();
            if (st != ERP_OK) return st;
            if (e != cudaSuccess) g.disabled = true;
            return body();
        }
        g.launches = ctx->launches - l0;
        ctx->launches = l0;
        g.key = k; g.key_gen = ctx->scratch_gen;
        memcpy(g.knn_stats, ctx->knn_stats, sizeof g.knn_stats);
        g.knn_bin = ctx->knn_bin;
        g.sc_misc_dev = ctx->sc_misc_dev; g.tc_misc_dev = ctx->tc_misc_dev; g.n_ev_score = ctx->n_ev_score;
        ERP_CUDA(cudaGraphLaunch(g.exec, ctx->stream));
        ctx->launches += g.launches;
        return ERP_OK;
    }
    const int st = body();
    g.seen = k; g.seen_gen = ctx->scratch_gen;
    return st;
}

// search + (multi-GPU: one 8-byte max all-reduce) + finish, everything enqueued, nothing awaited.
// k_ready: the correspondence operand of the tensor-core search was written by the gather.
int pose_chain_tail(erp_ctx* ctx, const double* dl, const double* dr, const float* dl4, const float* dr4, int m_cap, const int32_t* d_m,
                    uint64_t seed, uint64_t hyp_offset, int H, int S, int metric, float tau, bool k_ready, bool reduce,
                    uint8_t* d_mask, erp_ransac_result* d_res)
{
    int st = ERP_OK;
    uint64_t* d_packed = ctx->scratch<uint64_t>(S_PACKED, 4, &st);
    ERP_TRY(st);
    ERP_CUDA(cudaMemsetAsync(d_packed, 0, sizeof(uint64_t), ctx->stream));
    ERP_TRY(ransac_search(ctx, dl, dr, dl4, dr4, m_cap, d_m, seed, hyp_offset, H, S, metric, tau, k_ready, d_packed));
    if (reduce) ERP_TRY(comm_allreduce_best(ctx, d_packed));
    return ransac_finish(ctx, dl, dr, dl4, dr4, m_cap, d_m, seed, d_packed, S, metric, tau, d_mask, d_res);
}

// scratch of the chain for up to m_cap correspondences
int pose_chain_buffers(erp_ctx* ctx, int m_cap, PoseBuffers* b)
{
    int st = ERP_OK;
    b->l3 = ctx->scratch<double>(S_L3, (size_t)m_cap * 3 + 4, &st);
    b->r3 = ctx->scratch<double>(S_R3, (size_t)m_cap * 3 + 4, &st);
    b->l4 = ctx->scratch<float>(S_L4, (size_t)m_cap * 4 + 4, &st);
    b->r4 = ctx->scratch<float>(S_R4, (size_t)m_cap * 4 + 4, &st);
    b->mask = ctx->scratch<uint8_t>(S_MASK, (size_t)m_cap + 4, &st);
    b->res = ctx->scratch<erp_ransac_result>(S_RESULT, 1, &st);
    return st;
}

} // namespace erp

int erp::check_ransac_args(const char* who, erp_ctx* ctx, int H, int S, int metric, uint64_t hyp_offset)
{
    ERP_ARG(ctx && H >= 1, ERP_E_ARG, "%s: bad argument", who);
    ERP_ARG(S >= 8 && S <= 32, ERP_E_ARG, "%s: sample size must be in [8,32], got %d", who, S);
    ERP_ARG(metric >= 0 && metric <= 2, ERP_E_ARG, "%s: unknown metric %d", who, metric);
    ERP_ARG(hyp_offset + (uint64_t)H <= 0xFFFFFFFFull, ERP_E_LIMIT, "%s: hypothesis ids must fit 32 bits", who);
    return ERP_OK;
}

ERP_API int erp_ransac(erp_ctx* ctx, const double* l3, const double* r3, int m, uint64_t seed,
                       uint64_t hyp_offset, int H, int S, int metric, float tau,
                       erp_ransac_result* result, uint8_t* mask)
{
    ERP_ARG(result, ERP_E_ARG, "erp_ransac: result is null");
    ERP_TRY(check_ransac_args("erp_ransac", ctx, H, S, metric, hyp_offset));
    ERP_ARG(m >= S, ERP_E_TOO_FEW_POINTS, "erp_ransac: %d correspondences for sample size %d", m, S);
    DeviceGuard g(ctx->device);
    double *dl, *dr;
    float *dl4, *dr4;
    ERP_TRY(stage_bearings(ctx, l3, r3, m, &dl, &dr, &dl4, &dr4));
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, m, &b));
    ERP_TRY(pose_chain_tail(ctx, dl, dr, dl4, dr4, m, nullptr, seed, hyp_offset, H, S, metric, tau, false, false, b.mask, b.res));
    ERP_CUDA(cudaMemcpyAsync(result, b.res, sizeof *result, cudaMemcpyDeviceToHost, ctx->stream));
    if (mask) ERP_CUDA(cudaMemcpyAsync(mask, b.mask, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

ERP_API int erp_ransac_pixels(erp_ctx* ctx, int width, int height, const void* left_xy, const void* right_xy,
                              size_t stride_bytes, int m, uint64_t seed, uint64_t hyp_offset, int H, int S, int metric,
                              float tau, erp_ransac_result* result, uint8_t* mask)
{
    ERP_ARG(result && width > 0 && height > 0, ERP_E_ARG, "erp_ransac_pixels: bad argument");
    ERP_TRY(check_ransac_args("erp_ransac_pixels", ctx, H, S, metric, hyp_offset));
    ERP_ARG(stride_bytes >= 8 && stride_bytes % 4 == 0, ERP_E_ARG, "erp_ransac_pixels: bad stride %zu", stride_bytes);
    ERP_ARG(m >= S, ERP_E_TOO_FEW_POINTS, "erp_ransac_pixels: %d correspondences for sample size %d", m, S);
    ERP_ARG(left_xy && right_xy, ERP_E_ARG, "erp_ransac_pixels: null keypoints");
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    float* d_xy = ctx->scratch<float>(S_XY, (size_t)m * 4, &st);                 // left pairs, then right pairs
    ERP_TRY(st);
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, m, &b));
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy, left_xy, m, 8, stride_bytes));
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy + (size_t)m * 2, right_xy, m, 8, stride_bytes));
    const bool tc = ransac_uses_tc(ctx, H, m, metric);
    ScoreTcBuffers sb = {};
    if (tc) {
        ERP_TRY(score_tc_buffers(ctx, H < RANSAC_CHUNK ? H : RANSAC_CHUNK, m, &sb));
        ERP_CUDA(cudaMemsetAsync(sb.w, 0, W_WORDS_BYTES, ctx->stream));
    }
    ERP_TRY(bearings_pair_chain(ctx, d_xy, d_xy + (size_t)m * 2, 8, m, width, height, b.l3, b.r3, b.l4, b.r4, sb.Ks, sb.w));
    ERP_TRY(pose_chain_tail(ctx, b.l3, b.r3, b.l4, b.r4, m, nullptr, seed, hyp_offset, H, S, metric, tau, tc, false, b.mask, b.res));
    ERP_CUDA(cudaMemcpyAsync(result, b.res, sizeof *result, cudaMemcpyDeviceToHost, ctx->stream));
    if (mask) ERP_CUDA(cudaMemcpyAsync(mask, b.mask, (size_t)m, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}

// gather + bearings -> hypothesis search -> mask + refit on the device-resident match list of a pair (stage events 2, 3)
static int pose_after_match(erp_ctx* ctx, int nq, const PairArgs& a)
{
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, nq, &b));
    const bool tc = ransac_uses_tc(ctx, a.H, nq, a.metric);
    ScoreTcBuffers sb = {};
    if (tc) {
        ERP_TRY(score_tc_buffers(ctx, a.H < RANSAC_CHUNK ? a.H : RANSAC_CHUNK, nq, &sb));
        ERP_CUDA(cudaMemsetAsync(sb.w, 0, W_WORDS_BYTES, ctx->stream));
    }
    ERP_TRY(gather_bearings_chain(ctx, a.matches, nq, a.n_matches, a.left_xy, a.right_xy, a.kp_stride, 0, a.width, a.height,
                                  b.l3, b.r3, b.l4, b.r4, sb.Ks, sb.w));
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[2]));
    ERP_TRY(pose_chain_tail(ctx, b.l3, b.r3, b.l4, b.r4, nq, a.n_matches, a.seed, 0, a.H, a.S, a.metric, a.tau, tc, false,
                            a.mask ? a.mask : b.mask, a.result));
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[3]));
    return ERP_OK;
}

// the checks every pair call makes before its own
static int check_pair_args(const char* who, erp_ctx* ctx, RowKind k, int nq, int nt, const PairArgs& a)
{
    ERP_TRY(check_knn_args(who, ctx, nq, nt, k));
    ERP_TRY(check_ransac_args(who, ctx, a.H, a.S, a.metric, 0));
    ERP_ARG(a.matches && a.n_matches && a.result && a.width > 0 && a.height > 0, ERP_E_ARG, "%s: bad argument", who);
    ERP_ARG(a.left_xy && a.right_xy && a.kp_stride >= 8 && a.kp_stride % 4 == 0, ERP_E_ARG, "%s: bad keypoints", who);
    return ERP_OK;
}

static int pair_pose_dev(const char* who, erp_ctx* ctx, RowKind k, const void* d_q, int nq, const void* d_t, int nt, const PairArgs& a)
{
    ERP_TRY(check_pair_args(who, ctx, k, nq, nt, a));
    ERP_ARG(nq >= 1, ERP_E_TOO_FEW_POINTS, "%s: no query descriptors", who);
    DeviceGuard g(ctx->device);
    return graph_run(ctx, {k.bin ? PAIR_BIN : PAIR_F32, d_q, d_t, nq, nt, k.dim, a}, [&]() -> int {
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[0]));
    ERP_TRY(knn2_match_dev(who, ctx, k, d_q, nq, d_t, nt, a.ratio, a.cross_check, a.matches, a.n_matches));
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[1]));
    return pose_after_match(ctx, nq, a);
    });
}

int erp::pair_pose_download(erp_ctx* ctx, const char* who, cudaEvent_t ready, const PairArgs& dev, const PairArgs& out)
{
    // everything is enqueued: the host waits for the match list only (the pose chain keeps running), learns the match
    // count and brings the records back on the copy stream while the hypotheses are being scored
    int32_t n = 0;
    ERP_CUDA(cudaStreamWaitEvent(ctx->copy_stream, ready, 0));
    ERP_CUDA(cudaMemcpyAsync(&n, dev.n_matches, sizeof n, cudaMemcpyDeviceToHost, ctx->copy_stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    *out.n_matches = n;
    if (n > 0) ERP_CUDA(cudaMemcpyAsync(out.matches, dev.matches, sizeof(erp_dmatch) * (size_t)n, cudaMemcpyDeviceToHost, ctx->copy_stream));
    ERP_CUDA(cudaMemcpyAsync(out.result, dev.result, sizeof *out.result, cudaMemcpyDeviceToHost, ctx->stream));
    if (out.mask && n > 0) ERP_CUDA(cudaMemcpyAsync(out.mask, dev.mask, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->copy_stream));
    if (n < out.S) {
        set_error("%s: %d matches for sample size %d", who, n, out.S);
        return ERP_E_TOO_FEW_POINTS;
    }
    return ERP_OK;
}

static int pair_pose_host(const char* who, erp_ctx* ctx, RowKind k, const void* q, int nq, size_t qs, const void* t, int nt, size_t ts,
                          const PairArgs& a)
{
    ERP_TRY(check_pair_args(who, ctx, k, nq, nt, a));
    *a.n_matches = 0;
    ERP_ARG(nq >= 1, ERP_E_TOO_FEW_POINTS, "%s: no query descriptors", who);
    const size_t row = k.row_bytes();
    ERP_ARG(q && t && qs >= row && ts >= row, ERP_E_ARG, "%s: bad descriptor buffers", who);
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    PairArgs dev = a;
    dev.matches = ctx->scratch<erp_dmatch>(S_OUT, (size_t)nq, &st);
    dev.n_matches = ctx->scratch<int32_t>(S_NOUT, 4, &st);
    float* d_xy = ctx->scratch<float>(S_XY, ((size_t)nq + nt) * 2, &st);           // left pairs, then right pairs
    dev.left_xy = d_xy;
    dev.right_xy = d_xy + (size_t)nq * 2;
    dev.kp_stride = 8;
    uint8_t* dq = ctx->scratch<uint8_t>(S_Q, (size_t)nq * row + 16, &st);
    uint8_t* dt = ctx->scratch<uint8_t>(S_T, (size_t)nt * row + 16, &st);
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, nq, &b));
    ERP_TRY(st);
    dev.mask = b.mask;
    dev.result = b.res;
    int bounds[9];
    // binary pairs are not chunked: the cut of chunk_bounds was tuned for 256-byte float rows
    if (!k.bin && chunk_bounds(nq, nt, is_pageable(q), bounds) > 1) {
        // large pair: the descriptors travel in chunks behind the search (knn2_host), the keypoints follow on the copy
        // stream and are awaited by the gather; the chain is enqueued directly (launch cost hides behind the uploads)
        int32_t* idx2 = ctx->scratch<int32_t>(S_IDX2, (size_t)nq * 2 + 2, &st);
        float* dist2 = ctx->scratch<float>(S_DIST2, (size_t)nq * 2 + 2, &st);
        ERP_TRY(st);
        ERP_CUDA(record_timing(ctx, ctx->ev_stage[0]));
        ERP_TRY(knn2_host(ctx, k, q, nq, qs, t, nt, ts, idx2, dist2));
        ERP_TRY(upload_rows(ctx, ctx->copy_stream, d_xy, a.left_xy, nq, 8, a.kp_stride));
        ERP_TRY(upload_rows(ctx, ctx->copy_stream, d_xy + (size_t)nq * 2, a.right_xy, nt, 8, a.kp_stride));
        ERP_CUDA(cudaEventRecord(ctx->ev_copy[9], ctx->copy_stream));
        ERP_TRY(filter_matches(ctx, k, dq, nq, dt, nt, idx2, dist2, a.ratio, a.cross_check, dev.matches, dev.n_matches));
        ERP_CUDA(record_timing(ctx, ctx->ev_stage[1]));
        ERP_CUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_copy[9], 0));
        ERP_TRY(pose_after_match(ctx, nq, dev));
    } else {
        ERP_TRY(upload_rows(ctx, ctx->stream, dt, t, nt, row, ts));
        ERP_TRY(upload_rows(ctx, ctx->stream, dq, q, nq, row, qs));
        ERP_TRY(upload_rows(ctx, ctx->stream, d_xy, a.left_xy, nq, 8, a.kp_stride));
        ERP_TRY(upload_rows(ctx, ctx->stream, d_xy + (size_t)nq * 2, a.right_xy, nt, 8, a.kp_stride));
        ERP_TRY(pair_pose_dev(who, ctx, k, dq, nq, dt, nt, dev));
    }
    return pair_pose_download(ctx, who, ctx->ev_stage[1], dev, a);
}

ERP_API int erp_pair_pose_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim, float ratio, int cross_check,
                              const void* d_left_xy, const void* d_right_xy, size_t kp_stride_bytes, int width, int height,
                              uint64_t seed, int H, int S, int metric, float tau,
                              erp_dmatch* d_matches, int32_t* d_n_matches, uint8_t* d_mask, erp_ransac_result* d_result)
{
    return pair_pose_dev("erp_pair_pose_dev", ctx, RowKind::f32(dim), d_q, nq, d_t, nt,
                         {ratio, cross_check, d_left_xy, d_right_xy, kp_stride_bytes, width, height, seed, H, S, metric, tau,
                          d_matches, d_n_matches, d_mask, d_result});
}

ERP_API int erp_pair_pose(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                          int dim, float ratio, int cross_check,
                          const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                          uint64_t seed, int H, int S, int metric, float tau,
                          erp_dmatch* matches_out, int* n_matches, erp_ransac_result* result, uint8_t* mask)
{
    return pair_pose_host("erp_pair_pose", ctx, RowKind::f32(dim), q, nq, q_stride_bytes, t, nt, t_stride_bytes,
                          {ratio, cross_check, left_xy, right_xy, kp_stride_bytes, width, height, seed, H, S, metric, tau,
                           matches_out, n_matches, mask, result});
}

ERP_API int erp_pair_pose_bin_dev(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes, float ratio,
                                  int cross_check, const void* d_left_xy, const void* d_right_xy, size_t kp_stride_bytes, int width,
                                  int height, uint64_t seed, int H, int S, int metric, float tau,
                                  erp_dmatch* d_matches, int32_t* d_n_matches, uint8_t* d_mask, erp_ransac_result* d_result)
{
    return pair_pose_dev("erp_pair_pose_bin_dev", ctx, RowKind::binary(nbytes), d_q, nq, d_t, nt,
                         {ratio, cross_check, d_left_xy, d_right_xy, kp_stride_bytes, width, height, seed, H, S, metric, tau,
                          d_matches, d_n_matches, d_mask, d_result});
}

ERP_API int erp_pair_pose_bin(erp_ctx* ctx, const uint8_t* q, int nq, size_t q_stride_bytes, const uint8_t* t, int nt,
                              size_t t_stride_bytes, int nbytes, float ratio, int cross_check,
                              const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                              uint64_t seed, int H, int S, int metric, float tau,
                              erp_dmatch* matches_out, int* n_matches, erp_ransac_result* result, uint8_t* mask)
{
    return pair_pose_host("erp_pair_pose_bin", ctx, RowKind::binary(nbytes), q, nq, q_stride_bytes, t, nt, t_stride_bytes,
                          {ratio, cross_check, left_xy, right_xy, kp_stride_bytes, width, height, seed, H, S, metric, tau,
                           matches_out, n_matches, mask, result});
}

// ======================================================================================
// reference mode: initial_guess / find
// ======================================================================================
// glibc rand() (TYPE_3 additive feedback, r[i] = r[i-3] + r[i-31]) restated so the library
// neither reads nor disturbs the process-wide rand() state the way the reference does.
namespace {
struct GlibcRand {
    uint32_t r[34];
    int k = 0;
    explicit GlibcRand(unsigned seed)
    {
        int32_t w = (int32_t)(seed ? seed : 1);
        int32_t s[34];
        s[0] = w;
        for (int i = 1; i < 31; i++) {
            long hi = s[i - 1] / 127773, lo = s[i - 1] % 127773;
            long word = 16807 * lo - 2836 * hi;
            if (word < 0) word += 2147483647;
            s[i] = (int32_t)word;
        }
        for (int i = 31; i < 34; i++) s[i] = s[i - 31];
        for (int i = 0; i < 34; i++) r[i] = (uint32_t)s[i];
        for (int i = 0; i < 310; i++) next_raw();
    }
    uint32_t next_raw()
    {
        // ring of 34: new = r[k-31] + r[k-3]
        uint32_t v = r[(k + 34 - 31) % 34] + r[(k + 34 - 3) % 34];
        r[k % 34] = v;
        k = (k + 1) % 34;
        return v;
    }
    int next() { return (int)(next_raw() >> 1); }
};
} // namespace

ERP_API int erp_libstdcxx_sample_table(int m, int H, int S, unsigned seed, int32_t* table)
{
    ERP_ARG(m >= 1 && H >= 0 && S >= 0 && S <= m && table, ERP_E_ARG, "erp_libstdcxx_sample_table: bad argument");
    GlibcRand rng(seed);
    std::vector<int32_t> perm(m);
    for (int h = 0; h < H; h++) {
        // random_array::rand_idx_generate (src/eight_point.hpp:54-58): iota + random_shuffle;
        // libstdc++: for i in 1..n-1: swap(a[i], a[rand() % (i+1)])
        for (int i = 0; i < m; i++) perm[i] = i;
        for (int i = 1; i < m; i++) {
            int j = rng.next() % (i + 1);
            if (i != j) { int32_t t = perm[i]; perm[i] = perm[j]; perm[j] = t; }
        }
        memcpy(table + (size_t)h * S, perm.data(), sizeof(int32_t) * S);
    }
    return ERP_OK;
}

// initial_guess on bearings that are already on the device (dl, dr: m x 3 fp64)
static int initial_guess_dev(erp_ctx* ctx, const double* dl, const double* dr, int m,
                             const int32_t* samples, int H, int S,
                             float* R_vec_out, float* T_vec_out,
                             float* cand_R, float* cand_T, int* n_cand, int* chosen)
{
    ERP_ARG(ctx && R_vec_out && T_vec_out && H >= 1 && H <= 4096, ERP_E_ARG, "erp_initial_guess: bad argument");
    ERP_ARG(S >= 8 && m >= S, ERP_E_TOO_FEW_POINTS,
            "erp_initial_guess: sample size %d of %d correspondences (the reference needs match_size >= 32)", S, m);
    std::vector<int32_t> replay;
    if (!samples) {
        replay.resize((size_t)H * S);
        ERP_TRY(erp_libstdcxx_sample_table(m, H, S, 1, replay.data()));
        samples = replay.data();
    }
    int st = ERP_OK;
    float* dP = ctx->scratch<float>(S_POSE, (size_t)H * ERP_POSE_FLOATS + (size_t)H * 12 + 16, &st);
    ERP_TRY(st);
    // hypotheses solved exactly as erp_eight_point_batch does (pose included)
    for (size_t i = 0; i < (size_t)H * S; i++)
        ERP_ARG(samples[i] >= 0 && samples[i] < m, ERP_E_ARG, "sample index %d out of range [0,%d)", samples[i], m);
    int32_t* d_s = ctx->scratch<int32_t>(S_SAMPLES, (size_t)H * S, &st);
    double* dE = ctx->scratch<double>(S_E, (size_t)H * 9, &st);
    ERP_TRY(st);
    ERP_CUDA(cudaMemcpyAsync(d_s, samples, sizeof(int32_t) * (size_t)H * S, cudaMemcpyHostToDevice, ctx->stream));
    ERP_TRY(erp_eight_point_batch_dev(ctx, dl, dr, m, d_s, H, S, 0, 0, dE, dP));
    float* d_candR = dP + (size_t)H * ERP_POSE_FLOATS;
    float* d_candT = d_candR + (size_t)H * 6;
    int32_t* d_out = ctx->scratch<int32_t>(S_NOUT, 4, &st);
    ERP_TRY(st);
    ERP_TRY(consensus(ctx, dP, H, d_candR, d_candT, d_out));
    int32_t res[2] = {0, -1};
    ERP_CUDA(cudaMemcpyAsync(res, d_out, sizeof res, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    if (n_cand) *n_cand = res[0];
    if (chosen) *chosen = res[1];
    std::vector<float> hR((size_t)res[0] * 3 + 3), hT((size_t)res[0] * 3 + 3);
    if (res[0] > 0) {
        ERP_CUDA(cudaMemcpyAsync(hR.data(), d_candR, sizeof(float) * 3 * res[0], cudaMemcpyDeviceToHost, ctx->stream));
        ERP_CUDA(cudaMemcpyAsync(hT.data(), d_candT, sizeof(float) * 3 * res[0], cudaMemcpyDeviceToHost, ctx->stream));
        ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    }
    if (cand_R) memcpy(cand_R, hR.data(), sizeof(float) * 3 * res[0]);
    if (cand_T) memcpy(cand_T, hT.data(), sizeof(float) * 3 * res[0]);
    // the reference dereferences an empty vector here (src/eight_point.cpp:147-149): report it
    ERP_ARG(res[0] > 0 && res[1] >= 0, ERP_E_NO_CANDIDATE, "initial_guess: none of the %d hypotheses passed the <1.57 rad test", H);
    memcpy(R_vec_out, hR.data() + 3 * res[1], 12);
    memcpy(T_vec_out, hT.data() + 3 * res[1], 12);
    return ERP_OK;
}

ERP_API int erp_initial_guess(erp_ctx* ctx, const double* l3, const double* r3, int m,
                              const int32_t* samples, int H, int S,
                              float* R_vec_out, float* T_vec_out,
                              float* cand_R, float* cand_T, int* n_cand, int* chosen)
{
    ERP_ARG(ctx && m >= 0, ERP_E_ARG, "erp_initial_guess: bad argument");
    DeviceGuard g(ctx->device);
    double *dl, *dr;
    ERP_TRY(stage_bearings(ctx, l3, r3, m, &dl, &dr, nullptr, nullptr));
    return initial_guess_dev(ctx, dl, dr, m, samples, H, S, R_vec_out, T_vec_out, cand_R, cand_T, n_cand, chosen);
}

ERP_API int erp_find(erp_ctx* ctx, int width, int height, const void* left_xy, const void* right_xy,
                     size_t stride_bytes, int match_size, const int32_t* samples, int H, int S,
                     float* R_vec_out, float* T_vec_out)
{
    ERP_ARG(ctx && left_xy && right_xy && match_size >= 0, ERP_E_ARG, "erp_find: bad argument");
    if (H <= 0) H = 80;                               // src/eight_point.cpp:99
    if (S <= 0) S = (int)(match_size * 0.25);         // src/eight_point.cpp:102
    ERP_ARG(S >= 8, ERP_E_TOO_FEW_POINTS, "erp_find: match_size %d gives sample size %d < 8", match_size, S);
    ERP_ARG(width > 0 && height > 0 && stride_bytes >= 8 && stride_bytes % 4 == 0, ERP_E_ARG, "erp_find: bad image size or stride");
    // keypoints up once; the bearings (src/eight_point.cpp:163-186) never leave the device
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    float* d_xy = ctx->scratch<float>(S_XY, (size_t)match_size * 4, &st);
    ERP_TRY(st);
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, match_size, &b));
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy, left_xy, match_size, 8, stride_bytes));
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy + (size_t)match_size * 2, right_xy, match_size, 8, stride_bytes));
    ERP_TRY(bearings_pair_chain(ctx, d_xy, d_xy + (size_t)match_size * 2, 8, match_size, width, height, b.l3, b.r3, b.l4, b.r4,
                                nullptr, nullptr));
    return initial_guess_dev(ctx, b.l3, b.r3, match_size, samples, H, S, R_vec_out, T_vec_out, nullptr, nullptr, nullptr, nullptr);
}
