// dist.cu -- one ERP pair split over several B200s (SURVEY 8e / north_star): query rows and hypothesis ids per GPU,
// an all-gather of the per-rank match lists, ONE 8-byte max all-reduce of the packed best model, and a min all-reduce
// for cross-check.  NCCL over NVLink / NVSwitch; the library does not link NCCL, it dlopen()s libnccl.so.2 on first use
// (inside a torchrun rank that resolves to the copy torch already loaded, otherwise to the system one).
//
// Two cliques: erp_comm_init (one process per GPU, the caller distributes the unique id) and erp_group (one process,
// one worker thread per device, ncclCommInitAll): the collectives are tiny (8 B, <= 1.6 MB, 25.6 MB for the train
// all-gather of host-buffer calls), so a hand-written peer-memory kernel has nothing to overlap -- what matters is
// that nothing between them waits for the host (the match count stays on the device, common.cuh: RANSAC chain).
#include "score_common.cuh"

#include <dlfcn.h>
#include <nccl.h>   // types and prototypes only: every call goes through the table below

#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>

namespace erp {

constexpr int PEER_MAX = 64;

// ------------------------------------------------------------------------------------------ NCCL at run time
struct NcclApi {
    void* handle = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    std::string why;
};

static NcclApi load_nccl()
{
    NcclApi a;
    const char* names[] = {getenv("ERP_B200_NCCL"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
        if (!n || !*n) continue;
        a.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (a.handle) break;
        a.why = dlerror();
    }
    if (!a.handle) return a;
#define ERP_SYM(name) a.name = reinterpret_cast<decltype(a.name)>(dlsym(a.handle, "nccl" #name)); if (!a.name) { a.why = "symbol nccl" #name " missing"; a.handle = nullptr; return a; }
    ERP_SYM(GetUniqueId) ERP_SYM(CommInitRank) ERP_SYM(CommInitAll) ERP_SYM(CommDestroy) ERP_SYM(AllReduce) ERP_SYM(AllGather)
    ERP_SYM(GetErrorString) ERP_SYM(GetVersion)
#undef ERP_SYM
    return a;
}
static const NcclApi& nccl()
{
    static const NcclApi api = load_nccl();     // magic static: loaded once, thread safe
    return api;
}
static int need_nccl()
{
    if (nccl().handle) return ERP_OK;
    set_error("NCCL is not available (%s); multi-GPU calls need libnccl.so.2", nccl().why.c_str());
    return ERP_E_NCCL;
}
#define ERP_NCCL(call)                                                                              \
    do {                                                                                            \
        ncclResult_t r_ = (call);                                                                   \
        if (r_ != ncclSuccess) {                                                                    \
            erp::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, nccl().GetErrorString(r_)); \
            return ERP_E_NCCL;                                                                      \
        }                                                                                           \
    } while (0)

// ------------------------------------------------------------------------------------------ peer-memory exchange
// The two exchange steps of a sharded pair are tiny (<= 1.6 MB of match records, 8 bytes of best model) and sit on the
// critical path between kernels a few microseconds long: through NCCL they cost ~35 us each on this pool (plus the
// occasional millisecond when a proxy thread is descheduled).  Every rank therefore owns a WINDOW of device memory that
// all its peers map (cudaIpc* between processes, peer access inside one process) and the exchange is done by the
// library's own kernels over NVLink: a rank STORES its match slot / best word straight into every peer's window and
// then raises a per-source epoch flag there; consumers spin on flags in their own memory.  No kernel ever waits for
// something a peer has not been able to issue yet (every rank pushes before it waits), the epochs live on the device
// (a replayed CUDA graph advances them like a direct call), and spins are bounded (a protocol error traps instead of
// hanging the GPU).  NCCL stays for what is bandwidth bound or rare: the train-set all-gather of host-buffer calls,
// the cross-check reduction, and the window set-up itself.
struct WindowLayout {                     // byte offsets inside a window
    static constexpr size_t CTL = 0;             // uint32[64]: [0] epoch of the slot exchange, [1] of the best exchange, [2] ticket
    static constexpr size_t SLOT_FLAG = 256;     // uint32[64]: epoch of the last slot pushed by rank r
    static constexpr size_t BEST_FLAG = 512;     // uint32[64]
    static constexpr size_t BEST = 768;          // uint64[64]: packed best model of rank r
    static constexpr size_t SLOTS = 2048;        // erp_dmatch[nranks][slot_records]
};
struct WindowPtrs { uint8_t* peer[PEER_MAX]; };  // kernel argument: rank r's window as seen from this device

struct LocalClique {                      // one process, several devices (erp_group): pointers travel through host memory
    int n = 0;
    std::atomic<int> arrived{0}, phase{0};
    void* win[PEER_MAX] = {};
    int ok[PEER_MAX] = {};
    void barrier()
    {
        const int p = phase.load();
        if (arrived.fetch_add(1) + 1 == n) { arrived.store(0); phase.store(p + 1); }
        else while (phase.load() == p) std::this_thread::yield();
    }
};

struct Comm {
    ncclComm_t comm = nullptr;
    int nranks = 1, rank = 0;
    // peer window
    uint8_t* win = nullptr;
    size_t win_bytes = 0;
    WindowPtrs ptrs = {};
    bool opened[PEER_MAX] = {};          // cudaIpcOpenMemHandle mappings to close
    bool peer_failed = false;            // set once: stay on NCCL
    LocalClique* clique = nullptr;       // shared by the contexts of an erp_group (owned by the group)
};

static void window_close(Comm* c)
{
    for (int r = 0; r < c->nranks && r < PEER_MAX; r++) {
        if (c->opened[r] && c->ptrs.peer[r]) cudaIpcCloseMemHandle(c->ptrs.peer[r]);
        c->opened[r] = false;
        c->ptrs.peer[r] = nullptr;
    }
}

void comm_release(erp_ctx* ctx)
{
    if (!ctx->comm) return;
    graph_release(ctx);                  // a cached graph holds this clique's communicator and window pointers
    Comm* c = ctx->comm;
    window_close(c);
    if (c->win) cudaFree(c->win);
    if (c->comm && nccl().handle) nccl().CommDestroy(c->comm);
    delete c;
    ctx->comm = nullptr;
}

static inline int comm_size(const erp_ctx* ctx) { return ctx->comm ? ctx->comm->nranks : 1; }
static inline int comm_rank(const erp_ctx* ctx) { return ctx->comm ? ctx->comm->rank : 0; }

static inline void shard_range(int n, int rank, int world, int* lo, int* hi)
{
    const int base = n / world, rem = n % world;
    *lo = rank * base + (rank < rem ? rank : rem);
    *hi = *lo + base + (rank < rem ? 1 : 0);
}

// Collective: a window of at least `need` bytes on every rank, mapped by every rank.  Every rank of the clique calls it
// with the same size from the same call; returns null when the peer path is not available (then NCCL carries the
// exchange).  Growing re-does the set-up (host synchronisation: once per problem size, not per call).
static Comm* window_ensure(erp_ctx* ctx, size_t need)
{
    Comm* c = ctx->comm;
    static const bool off = [] { const char* e = getenv("ERP_B200_PEER"); return e && atoi(e) == 0; }();
    if (off || !c || c->peer_failed || c->nranks > PEER_MAX) return nullptr;
    if (c->win && c->win_bytes >= need) return c;
    if (ctx->capturing) return nullptr;                       // never during a capture: the first (direct) call sizes it
    const int G = c->nranks, rank = c->rank;
    size_t bytes = need < (size_t)(8 << 20) ? (size_t)(8 << 20) : need + need / 2;
    int good = 1;
    cudaStreamSynchronize(ctx->stream);
    if (c->clique) {
        // ---- one process: plain pointers, peer access was enabled when the group was made
        c->clique->barrier();                                 // nobody still uses the old windows
        if (c->win) { cudaFree(c->win); c->win = nullptr; }
        if (cudaMalloc(&c->win, bytes) != cudaSuccess || cudaMemset(c->win, 0, WindowLayout::SLOTS) != cudaSuccess) { cudaGetLastError(); good = 0; }
        c->clique->win[rank] = c->win;
        c->clique->ok[rank] = good;
        c->clique->barrier();
        for (int r = 0; r < G; r++) { good &= c->clique->ok[r]; c->ptrs.peer[r] = static_cast<uint8_t*>(c->clique->win[r]); }
        c->clique->barrier();                                 // everyone has read the table before it can change again
    } else {
        // ---- one process per GPU: cudaIpc handles, exchanged with NCCL
        int st = ERP_OK;
        uint8_t* xh = ctx->scratch<uint8_t>(S_GATHER, (size_t)G * 128 + 64, &st);
        if (st != ERP_OK) { c->peer_failed = true; return nullptr; }
        window_close(c);
        int32_t* flag = reinterpret_cast<int32_t*>(xh + (size_t)G * 128);
        // barrier: every rank has dropped its mappings before anyone frees the memory behind them
        if (nccl().AllReduce(flag, flag, 1, ncclInt32, ncclMin, c->comm, ctx->stream) != ncclSuccess || cudaStreamSynchronize(ctx->stream) != cudaSuccess) good = 0;
        if (c->win) { cudaFree(c->win); c->win = nullptr; }
        cudaIpcMemHandle_t mine;
        memset(&mine, 0, sizeof mine);
        if (cudaMalloc(&c->win, bytes) != cudaSuccess || cudaMemset(c->win, 0, WindowLayout::SLOTS) != cudaSuccess ||
            cudaIpcGetMemHandle(&mine, c->win) != cudaSuccess) { cudaGetLastError(); good = 0; }
        static_assert(sizeof(cudaIpcMemHandle_t) <= 128, "handle size");
        std::vector<uint8_t> all((size_t)G * 128, 0);
        cudaMemcpy(xh + (size_t)rank * 128, &mine, sizeof mine, cudaMemcpyHostToDevice);
        if (nccl().AllGather(xh + (size_t)rank * 128, xh, 128, ncclInt8, c->comm, ctx->stream) != ncclSuccess ||
            cudaMemcpyAsync(all.data(), xh, all.size(), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess) { cudaGetLastError(); good = 0; }
        for (int r = 0; r < G && good; r++) {
            if (r == rank) { c->ptrs.peer[r] = c->win; continue; }
            cudaIpcMemHandle_t h;
            memcpy(&h, all.data() + (size_t)r * 128, sizeof h);
            void* p = nullptr;
            if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); good = 0; break; }
            c->ptrs.peer[r] = static_cast<uint8_t*>(p);
            c->opened[r] = true;
        }
        // all or nothing: a rank that could not map a peer sends everybody back to NCCL
        int32_t mine_ok = good;
        cudaMemcpy(flag, &mine_ok, sizeof mine_ok, cudaMemcpyHostToDevice);
        if (nccl().AllReduce(flag, flag, 1, ncclInt32, ncclMin, c->comm, ctx->stream) != ncclSuccess ||
            cudaMemcpyAsync(&mine_ok, flag, sizeof mine_ok, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess) { cudaGetLastError(); mine_ok = 0; }
        good = mine_ok;
    }
    ctx->scratch_gen++;                                       // a cached graph holds window pointers
    if (!good) {
        window_close(c);
        if (c->win) { cudaFree(c->win); c->win = nullptr; }
        c->win_bytes = 0;
        c->peer_failed = true;
        return nullptr;
    }
    c->win_bytes = bytes;
    return c;
}

__device__ __forceinline__ void spin_until(const volatile uint32_t* flag, uint32_t epoch)
{
    if ((int32_t)(*flag - epoch) >= 0) return;
    const long long t0 = clock64();
    while ((int32_t)(*flag - epoch) < 0) {
        __nanosleep(40);
        if (clock64() - t0 > 8000000000LL) __trap();          // ~4 s: a peer never arrived
    }
}

// my match slot (header + records) into every peer's window, then the epoch flag of this rank on every peer
__global__ void __launch_bounds__(256)
push_slots_kernel(WindowPtrs w, int G, int rank, int slot_records)
{
    __shared__ int last;
    uint8_t* local = w.peer[rank];
    const int4* mine = reinterpret_cast<const int4*>(local + WindowLayout::SLOTS) + (size_t)rank * slot_records;
    const uint32_t epoch = reinterpret_cast<volatile uint32_t*>(local + WindowLayout::CTL)[0] + 1;
    int n = mine[0].x;                                         // header: the count the filter wrote
    n = n < 0 ? 0 : (n < slot_records - 1 ? n : slot_records - 1);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= n) {
        const int4 rec = mine[i];
        for (int p = 0; p < G; p++)
            if (p != rank) (reinterpret_cast<int4*>(w.peer[p] + WindowLayout::SLOTS) + (size_t)rank * slot_records)[i] = rec;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(reinterpret_cast<uint32_t*>(local + WindowLayout::CTL) + 2, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence_system();
    if (threadIdx.x < G) reinterpret_cast<volatile uint32_t*>(w.peer[threadIdx.x] + WindowLayout::SLOT_FLAG)[rank] = epoch;
    if (threadIdx.x == 0) reinterpret_cast<uint32_t*>(local + WindowLayout::CTL)[2] = 0;
}

// the single small reduction of north_star: every rank stores its packed best into every window, waits for the others'
// and keeps the maximum (count, then lowest hypothesis id).  One block.
__global__ void __launch_bounds__(PEER_MAX)
xchg_best_kernel(WindowPtrs w, int G, int rank, unsigned long long* __restrict__ packed)
{
    __shared__ unsigned long long red[PEER_MAX];
    uint8_t* local = w.peer[rank];
    const uint32_t epoch = reinterpret_cast<volatile uint32_t*>(local + WindowLayout::CTL)[1] + 1;
    const int r = threadIdx.x;
    const unsigned long long mine = *packed;
    unsigned long long v = 0;
    if (r < G) {
        reinterpret_cast<volatile unsigned long long*>(w.peer[r] + WindowLayout::BEST)[rank] = mine;
        __threadfence_system();
        reinterpret_cast<volatile uint32_t*>(w.peer[r] + WindowLayout::BEST_FLAG)[rank] = epoch;
        spin_until(reinterpret_cast<volatile uint32_t*>(local + WindowLayout::BEST_FLAG) + r, epoch);
        __threadfence_system();
        v = reinterpret_cast<volatile unsigned long long*>(local + WindowLayout::BEST)[r];
    }
    red[r] = v;
    __syncthreads();
    if (r == 0) {
        for (int i = 1; i < G; i++) v = red[i] > v ? red[i] : v;
        *packed = v;
        reinterpret_cast<volatile uint32_t*>(local + WindowLayout::CTL)[1] = epoch;
    }
}

int comm_allreduce_best(erp_ctx* ctx, uint64_t* d_packed)
{
    if (comm_size(ctx) == 1) return ERP_OK;
    if (Comm* c = window_ensure(ctx, WindowLayout::SLOTS)) {
        xchg_best_kernel<<<1, PEER_MAX, 0, ctx->stream>>>(c->ptrs, c->nranks, c->rank, reinterpret_cast<unsigned long long*>(d_packed));
        ERP_LAUNCH(ctx, "xchg_best_kernel");
        return ERP_OK;
    }
    // the packed word is < 2^63 (counts are < 2^31), unsigned max orders (count, then lowest id)
    ERP_NCCL(nccl().AllReduce(d_packed, d_packed, 1, ncclUint64, ncclMax, ctx->comm->comm, ctx->stream));
    return ERP_OK;
}

// candidates for the second reduction of the cross-check: my query id where I attain the global minimum
__global__ void cross_candidates_kernel(const double* __restrict__ mine_d2, const double* __restrict__ gmin_d2, int32_t* __restrict__ best_q, int nt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nt && !(mine_d2[i] == gmin_d2[i])) best_q[i] = 0x7fffffff;
}
__global__ void fill_reverse_kernel(int32_t* __restrict__ best_q, double* __restrict__ best_d2, int nt)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nt) { best_q[i] = 0x7fffffff; best_d2[i] = INFINITY; }
}

static int comm_cross_check(erp_ctx* ctx, int32_t* d_best_q, double* d_best_d2, int nt)
{
    if (comm_size(ctx) == 1 || nt == 0) return ERP_OK;
    int st = ERP_OK;
    double* gmin = ctx->scratch<double>(S_REVD2, (size_t)nt * 2, &st) + nt;
    ERP_TRY(st);
    ERP_NCCL(nccl().AllReduce(d_best_d2, gmin, (size_t)nt, ncclDouble, ncclMin, ctx->comm->comm, ctx->stream));
    cross_candidates_kernel<<<cdiv(nt, 256), 256, 0, ctx->stream>>>(d_best_d2, gmin, d_best_q, nt);
    ERP_LAUNCH(ctx, "cross_candidates_kernel");
    ERP_NCCL(nccl().AllReduce(d_best_q, d_best_q, (size_t)nt, ncclInt32, ncclMin, ctx->comm->comm, ctx->stream));
    ERP_CUDA(cudaMemcpyAsync(d_best_d2, gmin, sizeof(double) * (size_t)nt, cudaMemcpyDeviceToDevice, ctx->stream));
    return ERP_OK;
}

// this rank's rows of the query set against the whole train set: 2-NN, (reduced) cross-check, ratio filter.
// Matches carry global query ids.  d_out / d_n_out: device.
static int match_shard_dev(erp_ctx* ctx, const float* d_q_shard, int lo, int hi, const float* d_t, int nt, int dim, float ratio,
                           int cross_check, erp_dmatch* d_out, int32_t* d_n_out)
{
    const int nq = hi - lo;
    int st = ERP_OK;
    int32_t* idx2 = ctx->scratch<int32_t>(S_IDX2, (size_t)nq * 2 + 2, &st);
    float* dist2 = ctx->scratch<float>(S_DIST2, (size_t)nq * 2 + 2, &st);
    ERP_TRY(st);
    if (nq > 0) ERP_TRY(erp_knn2_dev(ctx, d_q_shard, nq, d_t, nt, dim, idx2, dist2, nullptr));
    int32_t* rev = nullptr;
    if (cross_check) {
        rev = ctx->scratch<int32_t>(S_REVQ, (size_t)nt, &st);
        double* rev_d2 = ctx->scratch<double>(S_REVD2, (size_t)nt * 2, &st);
        ERP_TRY(st);
        if (nq > 0) ERP_TRY(erp_nn1_reverse_dev(ctx, d_q_shard, nq, d_t, nt, dim, lo, rev, rev_d2));
        else {
            fill_reverse_kernel<<<cdiv(nt, 256), 256, 0, ctx->stream>>>(rev, rev_d2, nt);
            ERP_LAUNCH(ctx, "fill_reverse_kernel");
        }
        ERP_TRY(comm_cross_check(ctx, rev, rev_d2, nt));
    }
    return erp_match_filter_dev(ctx, idx2, dist2, nq, ratio, rev, lo, d_out, d_n_out);
}

} // namespace erp

using namespace erp;

// ======================================================================================
ERP_API int erp_shard_range(int n, int rank, int nranks, int* lo, int* hi)
{
    ERP_ARG(n >= 0 && nranks >= 1 && rank >= 0 && rank < nranks && lo && hi, ERP_E_ARG, "erp_shard_range: bad argument");
    shard_range(n, rank, nranks, lo, hi);
    return ERP_OK;
}

ERP_API int erp_comm_unique_id(void* id_out)
{
    ERP_ARG(id_out, ERP_E_ARG, "erp_comm_unique_id: null buffer");
    ERP_TRY(need_nccl());
    static_assert(sizeof(ncclUniqueId) == ERP_COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId id;
    ERP_NCCL(nccl().GetUniqueId(&id));
    memcpy(id_out, &id, sizeof id);
    return ERP_OK;
}

ERP_API int erp_comm_init(erp_ctx* ctx, int nranks, int rank, const void* id)
{
    ERP_ARG(ctx && id && nranks >= 1 && rank >= 0 && rank < nranks, ERP_E_ARG, "erp_comm_init: bad argument");
    ERP_ARG(nranks <= 64, ERP_E_LIMIT, "erp_comm_init: at most 64 ranks");
    comm_release(ctx);
    if (nranks == 1) return ERP_OK;
    ERP_TRY(need_nccl());
    DeviceGuard g(ctx->device);
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof uid);
    Comm* c = new Comm();
    c->nranks = nranks; c->rank = rank;
    ncclResult_t r = nccl().CommInitRank(&c->comm, nranks, uid, rank);
    if (r != ncclSuccess) {
        set_error("ncclCommInitRank(rank %d of %d) -> %s", rank, nranks, nccl().GetErrorString(r));
        delete c;
        return ERP_E_NCCL;
    }
    ctx->comm = c;
    return ERP_OK;
}

ERP_API int erp_comm_destroy(erp_ctx* ctx)
{
    ERP_ARG(ctx, ERP_E_ARG, "erp_comm_destroy: null context");
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    comm_release(ctx);
    return ERP_OK;
}

ERP_API int erp_comm_size(erp_ctx* ctx) { return ctx ? comm_size(ctx) : 0; }
ERP_API int erp_comm_rank(erp_ctx* ctx) { return ctx ? comm_rank(ctx) : -1; }

ERP_API int erp_comm_allreduce_best_dev(erp_ctx* ctx, uint64_t* d_packed)
{
    ERP_ARG(ctx && d_packed, ERP_E_ARG, "erp_comm_allreduce_best_dev: bad argument");
    DeviceGuard g(ctx->device);
    return comm_allreduce_best(ctx, d_packed);
}

ERP_API int erp_comm_cross_check_dev(erp_ctx* ctx, int32_t* d_best_q, double* d_best_d2, int nt)
{
    ERP_ARG(ctx && d_best_q && d_best_d2 && nt >= 0, ERP_E_ARG, "erp_comm_cross_check_dev: bad argument");
    DeviceGuard g(ctx->device);
    return comm_cross_check(ctx, d_best_q, d_best_d2, nt);
}

// the sharded pair on G > 1 ranks: checks, then match -> exchange -> gather -> hypothesis search -> mask + refit
static int pair_pose_dist_dev(erp_ctx* ctx, const float* d_q_shard, int nq_total, const float* d_t, int nt, int dim, const PairArgs& a)
{
    const char* who = "erp_pair_pose_dist_dev";
    const int G = comm_size(ctx), rank = comm_rank(ctx);
    ERP_ARG(nq_total >= 1 && nt >= 2, ERP_E_TOO_FEW_TRAIN, "%s: nq %d, nt %d", who, nq_total, nt);
    ERP_TRY(RowKind::f32(dim).check_dim(who));
    ERP_ARG(d_t && a.matches && a.n_matches && a.result && a.width > 0 && a.height > 0, ERP_E_ARG, "%s: bad argument", who);
    ERP_ARG(a.left_xy && a.right_xy && a.kp_stride >= 8 && a.kp_stride % 4 == 0, ERP_E_ARG, "%s: bad keypoints", who);
    ERP_TRY(check_ransac_args(who, ctx, a.H, a.S, a.metric, 0));
    ERP_ARG(a.H >= G, ERP_E_ARG, "%s: %d hypotheses for %d ranks", who, a.H, G);
    DeviceGuard g(ctx->device);
    int lo, hi, hlo, hhi;
    shard_range(nq_total, rank, G, &lo, &hi);
    shard_range(a.H, rank, G, &hlo, &hhi);
    ERP_ARG(hi == lo || d_q_shard, ERP_E_ARG, "%s: null query shard", who);
    // slots of the match exchange: [header | up to cap records] per rank, in the peer window when there is one
    const int cap = cdiv(nq_total, G), slot = cap + 1;
    Comm* win = window_ensure(ctx, WindowLayout::SLOTS + (size_t)slot * G * sizeof(erp_dmatch));
    return graph_run(ctx, {PAIR_DIST, d_q_shard, d_t, nq_total, nt, dim, a}, [&]() -> int {
    int st = ERP_OK;
    erp_dmatch* slots = win ? reinterpret_cast<erp_dmatch*>(win->win + WindowLayout::SLOTS)
                            : ctx->scratch<erp_dmatch>(S_XCHG, (size_t)slot * G, &st);
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, nq_total, &b));
    const bool tc = ransac_uses_tc(ctx, hhi - hlo, nq_total, a.metric);
    ScoreTcBuffers sb = {};
    if (tc) ERP_TRY(score_tc_buffers(ctx, (hhi - hlo) < RANSAC_CHUNK ? (hhi - hlo) : RANSAC_CHUNK, nq_total, &sb));
    ERP_TRY(st);
    erp_dmatch* mine = slots + (size_t)slot * rank;

    ERP_CUDA(record_timing(ctx, ctx->ev_stage[0]));
    ERP_CUDA(cudaMemsetAsync(mine, 0, sizeof(erp_dmatch), ctx->stream));
    ERP_TRY(match_shard_dev(ctx, d_q_shard, lo, hi, d_t, nt, dim, a.ratio, a.cross_check, mine + 1, &mine->queryIdx));
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[1]));
    if (win) {
        // peer stores over NVLink + epoch flags; the gather below waits for the flags of all ranks
        push_slots_kernel<<<cdiv(slot, 256), 256, 0, ctx->stream>>>(win->ptrs, G, rank, slot);
        ERP_LAUNCH(ctx, "push_slots_kernel");
    } else {
        // in place: rank r's slot is already at its position of the receive buffer
        ERP_NCCL(nccl().AllGather(mine, slots, (size_t)slot * sizeof(erp_dmatch), ncclInt8, ctx->comm->comm, ctx->stream));
    }
    if (tc) ERP_CUDA(cudaMemsetAsync(sb.w, 0, W_WORDS_BYTES, ctx->stream));
    ERP_TRY(gather_slots_chain(ctx, slots, G, slot, nq_total, a.matches, a.n_matches, a.left_xy, a.right_xy, a.kp_stride,
                               a.width, a.height, b.l3, b.r3, b.l4, b.r4, sb.Ks, sb.w,
                               win ? reinterpret_cast<uint32_t*>(win->win + WindowLayout::CTL) : nullptr,
                               win ? reinterpret_cast<uint32_t*>(win->win + WindowLayout::SLOT_FLAG) : nullptr));
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[2]));
    ERP_TRY(pose_chain_tail(ctx, b.l3, b.r3, b.l4, b.r4, nq_total, a.n_matches, a.seed, (uint64_t)hlo, hhi - hlo, a.S, a.metric, a.tau, tc,
                            true, a.mask ? a.mask : b.mask, a.result));
    ERP_CUDA(record_timing(ctx, ctx->ev_stage[3]));
    return ERP_OK;
    });
}

ERP_API int erp_pair_pose_dist_dev(erp_ctx* ctx, const float* d_q_shard, int nq_total, const float* d_t, int nt, int dim,
                                   float ratio, int cross_check,
                                   const void* d_left_xy, const void* d_right_xy, size_t kp_stride_bytes, int width, int height,
                                   uint64_t seed, int H_total, int S, int metric, float tau,
                                   erp_dmatch* d_matches, int32_t* d_n_matches, uint8_t* d_mask, erp_ransac_result* d_result)
{
    ERP_ARG(ctx, ERP_E_ARG, "erp_pair_pose_dist_dev: null context");
    if (comm_size(ctx) == 1)
        return erp_pair_pose_dev(ctx, d_q_shard, nq_total, d_t, nt, dim, ratio, cross_check, d_left_xy, d_right_xy, kp_stride_bytes,
                                 width, height, seed, H_total, S, metric, tau, d_matches, d_n_matches, d_mask, d_result);
    return pair_pose_dist_dev(ctx, d_q_shard, nq_total, d_t, nt, dim,
                              {ratio, cross_check, d_left_xy, d_right_xy, kp_stride_bytes, width, height, seed, H_total, S, metric, tau,
                               d_matches, d_n_matches, d_mask, d_result});
}

namespace erp {

// upload of one rank's share for a host-buffer call: the query shard, 1/G of the train rows (then all-gathered over
// NVLink into the replicated train set) -- G times less PCIe traffic per GPU than uploading everything everywhere
static int upload_sharded(erp_ctx* ctx, const float* q, int lo, int hi, size_t qs, const float* t, int nt, size_t ts, int dim,
                          float** dq_out, float** dt_out)
{
    const int G = comm_size(ctx), rank = comm_rank(ctx);
    const size_t row = (size_t)dim * sizeof(float);
    const int tcap = cdiv(nt, G);                    // train rows per rank in the all-gather (the last block may be short)
    int st = ERP_OK;
    float* dq = ctx->scratch<float>(S_Q, (size_t)(hi - lo) * dim + 4, &st);
    float* dt = ctx->scratch<float>(S_T, (size_t)tcap * G * dim + 4, &st);
    ERP_TRY(st);
    ERP_TRY(upload_rows(ctx, ctx->stream, dq, reinterpret_cast<const char*>(q) + (size_t)lo * qs, hi - lo, row, qs));
    const int t0 = rank * tcap < nt ? rank * tcap : nt, t1 = (rank + 1) * tcap < nt ? (rank + 1) * tcap : nt;
    ERP_TRY(upload_rows(ctx, ctx->stream, dt + (size_t)t0 * dim, reinterpret_cast<const char*>(t) + (size_t)t0 * ts, t1 - t0, row, ts));
    if (G > 1)
        ERP_NCCL(nccl().AllGather(dt + (size_t)rank * tcap * dim, dt, (size_t)tcap * dim, ncclFloat, ctx->comm->comm, ctx->stream));
    *dq_out = dq; *dt_out = dt;
    return ERP_OK;
}

} // namespace erp

ERP_API int erp_pair_pose_dist(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                               int dim, float ratio, int cross_check,
                               const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                               uint64_t seed, int H, int S, int metric, float tau,
                               erp_dmatch* matches_out, int* n_matches, erp_ransac_result* result, uint8_t* mask)
{
    ERP_ARG(ctx, ERP_E_ARG, "erp_pair_pose_dist: null context");
    if (comm_size(ctx) == 1)
        return erp_pair_pose(ctx, q, nq, q_stride_bytes, t, nt, t_stride_bytes, dim, ratio, cross_check, left_xy, right_xy,
                             kp_stride_bytes, width, height, seed, H, S, metric, tau, matches_out, n_matches, result, mask);
    ERP_ARG(n_matches && result && matches_out && q && t && left_xy && right_xy, ERP_E_ARG, "erp_pair_pose_dist: null argument");
    *n_matches = 0;
    ERP_ARG(nq >= 1 && nt >= 2, ERP_E_TOO_FEW_TRAIN, "erp_pair_pose_dist: nq %d, nt %d", nq, nt);
    ERP_TRY(RowKind::f32(dim).check_dim("erp_pair_pose_dist"));
    const size_t row = (size_t)dim * sizeof(float);
    ERP_ARG(q_stride_bytes >= row && t_stride_bytes >= row && kp_stride_bytes >= 8 && kp_stride_bytes % 4 == 0, ERP_E_ARG,
            "erp_pair_pose_dist: bad stride");
    DeviceGuard g(ctx->device);
    const PairArgs out = {ratio, cross_check, left_xy, right_xy, kp_stride_bytes, width, height, seed, H, S, metric, tau,
                          matches_out, n_matches, mask, result};
    PairArgs dev = out;
    const int G = comm_size(ctx), rank = comm_rank(ctx);
    int lo, hi;
    shard_range(nq, rank, G, &lo, &hi);
    int st = ERP_OK;
    dev.matches = ctx->scratch<erp_dmatch>(S_OUT, (size_t)nq, &st);
    dev.n_matches = ctx->scratch<int32_t>(S_NOUT, 4, &st);
    float* d_xy = ctx->scratch<float>(S_XY, ((size_t)nq + nt) * 2, &st);
    dev.left_xy = d_xy;
    dev.right_xy = d_xy + (size_t)nq * 2;
    dev.kp_stride = 8;
    PoseBuffers b;
    ERP_TRY(pose_chain_buffers(ctx, nq, &b));
    ERP_TRY(st);
    dev.mask = b.mask;
    dev.result = b.res;
    float *dq, *dt;
    ERP_TRY(upload_sharded(ctx, q, lo, hi, q_stride_bytes, t, nt, t_stride_bytes, dim, &dq, &dt));
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy, left_xy, nq, 8, kp_stride_bytes));
    ERP_TRY(upload_rows(ctx, ctx->stream, d_xy + (size_t)nq * 2, right_xy, nt, 8, kp_stride_bytes));
    ERP_TRY(pair_pose_dist_dev(ctx, dq, nq, dt, nt, dim, dev));
    // the host waits for the exchange only; the records come back while the hypotheses are being scored
    return pair_pose_download(ctx, "erp_pair_pose_dist", ctx->ev_stage[2], dev, out);
}

ERP_API int erp_knn2_match_dist(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                                int dim, float ratio, int cross_check, erp_dmatch* out, int* n_out)
{
    ERP_ARG(ctx, ERP_E_ARG, "erp_knn2_match_dist: null context");
    if (comm_size(ctx) == 1) return erp_knn2_match(ctx, q, nq, q_stride_bytes, t, nt, t_stride_bytes, dim, ratio, cross_check, out, n_out);
    ERP_ARG(n_out, ERP_E_ARG, "erp_knn2_match_dist: n_out is null");
    *n_out = 0;
    ERP_TRY(check_knn_args("erp_knn2_match_dist", ctx, nq, nt, RowKind::f32(dim)));
    if (nq == 0) return ERP_OK;
    const size_t row = (size_t)dim * sizeof(float);
    ERP_ARG(q && t && q_stride_bytes >= row && t_stride_bytes >= row, ERP_E_ARG, "erp_knn2_match_dist: bad descriptor buffers");
    DeviceGuard g(ctx->device);
    int lo, hi;
    shard_range(nq, comm_rank(ctx), comm_size(ctx), &lo, &hi);
    ERP_ARG(hi == lo || out, ERP_E_ARG, "erp_knn2_match_dist: out is null");
    int st = ERP_OK;
    erp_dmatch* d_out = ctx->scratch<erp_dmatch>(S_OUT, (size_t)(hi - lo) + 1, &st);
    int32_t* d_n = ctx->scratch<int32_t>(S_NOUT, 4, &st);
    ERP_TRY(st);
    float *dq, *dt;
    ERP_TRY(upload_sharded(ctx, q, lo, hi, q_stride_bytes, t, nt, t_stride_bytes, dim, &dq, &dt));
    ERP_TRY(match_shard_dev(ctx, dq, lo, hi, dt, nt, dim, ratio, cross_check, d_out, d_n));
    return download_matches(ctx, d_out, d_n, (size_t)(hi - lo), out, n_out);
}

ERP_API int erp_knn2_match_dist_dev(erp_ctx* ctx, const float* d_q_shard, int nq_total, const float* d_t, int nt, int dim,
                                    float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out)
{
    ERP_ARG(ctx && d_n_out, ERP_E_ARG, "erp_knn2_match_dist_dev: bad argument");
    ERP_TRY(check_knn_args("erp_knn2_match_dist_dev", ctx, nq_total, nt, RowKind::f32(dim)));
    DeviceGuard g(ctx->device);
    int lo, hi;
    shard_range(nq_total, comm_rank(ctx), comm_size(ctx), &lo, &hi);
    ERP_ARG(hi == lo || (d_q_shard && d_t && d_out), ERP_E_ARG, "erp_knn2_match_dist_dev: null buffer");
    return match_shard_dev(ctx, d_q_shard, lo, hi, d_t, nt, dim, ratio, cross_check, d_out, d_n_out);
}

// ======================================================================================
// one process, several devices: contexts + clique + one worker thread per device
// ======================================================================================
struct erp_group {
    erp::LocalClique clique;              // host-side rendezvous of the peer windows (one process: no cudaIpc)
    std::vector<erp_ctx*> ctx;
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    std::function<int(int)> job;
    uint64_t generation = 0;
    int pending = 0;
    bool stop = false;
    std::vector<int> status;
    std::vector<std::string> error;

    void worker(int rank)
    {
        uint64_t seen = 0;
        for (;;) {
            std::function<int(int)> fn;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_job.wait(lk, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
                fn = job;
            }
            int st = fn(rank);
            std::string msg = st != ERP_OK ? erp_last_error() : "";
            {
                std::lock_guard<std::mutex> lk(mu);
                status[rank] = st;
                error[rank] = msg;
                if (--pending == 0) cv_done.notify_all();
            }
        }
    }
    // runs fn(rank) on every worker; first failing rank's status and message are reported to the caller
    int run(std::function<int(int)> fn)
    {
        {
            std::lock_guard<std::mutex> lk(mu);
            job = std::move(fn);
            pending = (int)ctx.size();
            generation++;
        }
        cv_job.notify_all();
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return pending == 0; });
        for (size_t r = 0; r < ctx.size(); r++)
            if (status[r] != ERP_OK) {
                set_error("rank %zu: %s", r, error[r].c_str());
                return status[r];
            }
        return ERP_OK;
    }
};

ERP_API void erp_group_destroy(erp_group* g)
{
    if (!g) return;
    {
        std::lock_guard<std::mutex> lk(g->mu);
        g->stop = true;
    }
    g->cv_job.notify_all();
    for (auto& t : g->workers) if (t.joinable()) t.join();
    for (erp_ctx* c : g->ctx) if (c) erp_ctx_destroy(c);
    delete g;
}

ERP_API int erp_group_create(const int* devices, int ndev, erp_group** out)
{
    ERP_ARG(out, ERP_E_ARG, "erp_group_create: out is null");
    *out = nullptr;
    ERP_ARG(devices && ndev >= 1 && ndev <= 64, ERP_E_ARG, "erp_group_create: 1..64 devices");
    for (int i = 0; i < ndev; i++)
        for (int j = 0; j < i; j++) ERP_ARG(devices[i] != devices[j], ERP_E_ARG, "erp_group_create: device %d listed twice", devices[i]);
    if (ndev > 1) ERP_TRY(need_nccl());
    erp_group* g = new erp_group();
    g->ctx.assign(ndev, nullptr);
    g->status.assign(ndev, ERP_OK);
    g->error.assign(ndev, "");
    for (int i = 0; i < ndev; i++) {
        int st = erp_ctx_create(devices[i], &g->ctx[i]);
        if (st != ERP_OK) { erp_group_destroy(g); return st; }
    }
    if (ndev > 1) {
        std::vector<ncclComm_t> comms(ndev);
        ncclResult_t r = nccl().CommInitAll(comms.data(), ndev, devices);
        if (r != ncclSuccess) {
            set_error("ncclCommInitAll over %d devices -> %s", ndev, nccl().GetErrorString(r));
            erp_group_destroy(g);
            return ERP_E_NCCL;
        }
        // peer access for the windows (dist.cu: peer-memory exchange); without it the exchange stays on NCCL
        bool p2p = true;
        for (int i = 0; i < ndev && p2p; i++) {
            DeviceGuard dg(devices[i]);
            for (int j = 0; j < ndev && p2p; j++) {
                if (i == j) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, devices[i], devices[j]) != cudaSuccess || !can) { p2p = false; break; }
                cudaError_t e = cudaDeviceEnablePeerAccess(devices[j], 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) p2p = false;
                cudaGetLastError();
            }
        }
        g->clique.n = ndev;
        for (int i = 0; i < ndev; i++) {
            Comm* c = new Comm();
            c->comm = comms[i]; c->nranks = ndev; c->rank = i;
            c->clique = &g->clique;
            c->peer_failed = !p2p;
            g->ctx[i]->comm = c;
        }
    }
    for (int i = 0; i < ndev; i++) g->workers.emplace_back([g, i] { g->worker(i); });
    *out = g;
    return ERP_OK;
}

ERP_API int erp_group_size(erp_group* g) { return g ? (int)g->ctx.size() : 0; }
ERP_API erp_ctx* erp_group_ctx(erp_group* g, int rank) { return g && rank >= 0 && rank < (int)g->ctx.size() ? g->ctx[rank] : nullptr; }

ERP_API int erp_group_pair_pose(erp_group* g, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                                int dim, float ratio, int cross_check,
                                const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                                uint64_t seed, int H, int S, int metric, float tau,
                                erp_dmatch* matches_out, int* n_matches, erp_ransac_result* result, uint8_t* mask)
{
    ERP_ARG(g && n_matches && result && matches_out, ERP_E_ARG, "erp_group_pair_pose: bad argument");
    const int G = (int)g->ctx.size();
    // every rank ends with the same records; rank 0 writes the caller's buffers, the others a scratch of their own
    std::vector<std::vector<erp_dmatch>> other(G);
    std::vector<erp_ransac_result> res(G);
    std::vector<int> n(G, 0);
    int st = g->run([&](int r) {
        if (r != 0) other[r].resize((size_t)(nq > 0 ? nq : 1));
        return erp_pair_pose_dist(g->ctx[r], q, nq, q_stride_bytes, t, nt, t_stride_bytes, dim, ratio, cross_check, left_xy, right_xy,
                                  kp_stride_bytes, width, height, seed, H, S, metric, tau,
                                  r == 0 ? matches_out : other[r].data(), &n[r], &res[r], r == 0 ? mask : nullptr);
    });
    *n_matches = n[0];
    *result = res[0];
    return st;
}

ERP_API int erp_group_knn2_match(erp_group* g, const float* q, int nq, size_t q_stride_bytes,
                                 const float* t, int nt, size_t t_stride_bytes, int dim,
                                 float ratio, int cross_check, erp_dmatch* out, int* n_out)
{
    ERP_ARG(g && n_out, ERP_E_ARG, "erp_group_knn2_match: bad argument");
    *n_out = 0;
    const int G = (int)g->ctx.size();
    if (G == 1) return erp_knn2_match(g->ctx[0], q, nq, q_stride_bytes, t, nt, t_stride_bytes, dim, ratio, cross_check, out, n_out);
    ERP_ARG(nq == 0 || out, ERP_E_ARG, "erp_group_knn2_match: out is null");
    // rank r's part lands at its shard offset of the caller's buffer (a shard never yields more records than rows) and is
    // then moved down to close the gaps: rank order keeps ascending queryIdx
    std::vector<int> n(G, 0), lo(G, 0), hi(G, 0);
    for (int r = 0; r < G; r++) shard_range(nq > 0 ? nq : 0, r, G, &lo[r], &hi[r]);
    int st = g->run([&](int r) {
        return erp_knn2_match_dist(g->ctx[r], q, nq, q_stride_bytes, t, nt, t_stride_bytes, dim, ratio, cross_check,
                                   out ? out + lo[r] : nullptr, &n[r]);
    });
    ERP_TRY(st);
    int total = 0;
    for (int r = 0; r < G; r++) {
        if (n[r] > 0 && total != lo[r]) memmove(out + total, out + lo[r], sizeof(erp_dmatch) * (size_t)n[r]);
        total += n[r];
    }
    *n_out = total;
    return ERP_OK;
}
