// geometry.cu -- pixel->bearing, Philox minimal samples, batched eight-point solve,
// consensus pick.  Replaces /root/reference/src/eight_point.cpp:16-192 on the device.
//
// The solve is the Gram form of OpenCV's one-sided Jacobi SVD: cv::SVDecomp(A) rotates the
// columns of the S x 9 matrix A (modules/core/src/lapack.cpp, JacobiSVDImpl_); the rotation of
// columns (i,j) depends only on a = |a_i|^2, b = |a_j|^2, p = a_i.a_j, i.e. on the 9 x 9 Gram
// matrix G = A^T A.  Applying the same cyclic pivot order and the same (c,s) formulas to G
// (G <- J^T G J, V <- V J) reproduces the same right singular vectors, including their sign,
// without ever materialising A: S x 9 collapses to 45 doubles per hypothesis, which is what
// lets a million hypotheses run concurrently.  The 3 x 3 SVDs (rank-2 projection and
// cv::decomposeEssentialMat) are run one-sided exactly as OpenCV does.
#include "score_common.cuh"

#include <float.h>

namespace erp {

// ------------------------------------------------------------------ bearings (eight_point.cpp:163-186)
__global__ void bearings_kernel(const char* __restrict__ xy, size_t stride, int n, int W, int H,
                                double* __restrict__ out3, float4* __restrict__ out4)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* p = reinterpret_cast<const float*>(xy + (size_t)i * stride);
    float fx = __fdiv_rn(p[0], (float)W);      // float quotient, then promoted (pt.x / im_width)
    float fy = __fdiv_rn(p[1], (float)H);
    double lon = 2 * 3.14159265358979323846 * (double)fx;
    double lat = 3.14159265358979323846 * (double)fy;
    double sl, cl, so, co;
    sincos(lat, &sl, &cl);
    sincos(lon, &so, &co);
    double x = -sl * co, y = sl * so, z = cl;   // MPEG OMAF axes
    if (out3) { out3[3 * (size_t)i] = x; out3[3 * (size_t)i + 1] = y; out3[3 * (size_t)i + 2] = z; }
    if (out4) out4[i] = make_float4((float)x, (float)y, (float)z, 0.f);
}

__device__ __forceinline__ void pixel_to_bearing(const float* p, int W, int H, double& x, double& y, double& z)
{
    float fx = __fdiv_rn(p[0], (float)W), fy = __fdiv_rn(p[1], (float)H);
    double lon = 2 * 3.14159265358979323846 * (double)fx, lat = 3.14159265358979323846 * (double)fy;
    double sl, cl, so, co;
    sincos(lat, &sl, &cl);
    sincos(lon, &so, &co);
    x = -sl * co; y = sl * so; z = cl;
}

// spherical_surf.cpp:155-162 (gather the matched keypoints) fused with eight_point.cpp:163-186.  The match count may live
// on the device (n_dev; the launch covers n_cap slots).  With Ks the same pass also writes the correspondence operand of
// the tensor-core hypothesis search and its m-dependent words (score_common.cuh: prep_k_slot) -- launched with whole warps.
__global__ void gather_bearings_kernel(const erp_dmatch* __restrict__ mt, int n_cap, const int32_t* __restrict__ n_dev,
                                       const char* __restrict__ lxy, const char* __restrict__ rxy, size_t stride, int q_offset,
                                       int W, int H, double* __restrict__ l3, double* __restrict__ r3,
                                       float4* __restrict__ l4, float4* __restrict__ r4, float* __restrict__ Ks, int32_t* __restrict__ w)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = dev_len(n_dev, n_cap);
    float4 lf = make_float4(0.f, 0.f, 0.f, 0.f), rf = lf;
    if (i < n) {
        erp_dmatch m = mt[i];
        double x, y, z;
        pixel_to_bearing(reinterpret_cast<const float*>(lxy + (size_t)(m.queryIdx - q_offset) * stride), W, H, x, y, z);
        if (l3) { l3[3 * (size_t)i] = x; l3[3 * (size_t)i + 1] = y; l3[3 * (size_t)i + 2] = z; }
        lf = make_float4((float)x, (float)y, (float)z, 0.f);
        if (l4) l4[i] = lf;
        pixel_to_bearing(reinterpret_cast<const float*>(rxy + (size_t)m.trainIdx * stride), W, H, x, y, z);
        if (r3) { r3[3 * (size_t)i] = x; r3[3 * (size_t)i + 1] = y; r3[3 * (size_t)i + 2] = z; }
        rf = make_float4((float)x, (float)y, (float)z, 0.f);
        if (r4) r4[i] = rf;
    }
    if (Ks) prep_k_slot(i, n, lf, rf, Ks, w);
}

// Multi-GPU form: the per-rank match lists arrive in fixed-size slots (all-gather; record 0 of a slot is a header whose
// queryIdx holds the rank's count, the matches follow and already carry GLOBAL query ids).  This pass concatenates them
// in rank order (= ascending queryIdx, feature_matcher.cpp:50-56) into `out`, publishes the total, and does the
// gather + bearings + operand rows of gather_bearings_kernel on the fly.
constexpr int GATHER_MAX_RANKS = 64;
__global__ void gather_slots_kernel(const erp_dmatch* __restrict__ slots, int n_ranks, int slot_records, int n_cap,
                                    erp_dmatch* __restrict__ out, int32_t* __restrict__ n_out,
                                    const char* __restrict__ lxy, const char* __restrict__ rxy, size_t stride,
                                    int W, int H, double* __restrict__ l3, double* __restrict__ r3,
                                    float4* __restrict__ l4, float4* __restrict__ r4, float* __restrict__ Ks, int32_t* __restrict__ w,
                                    uint32_t* __restrict__ ctl, const uint32_t* __restrict__ slot_flag)
{
    __shared__ int prefix[GATHER_MAX_RANKS + 1];
    __shared__ int last;
    // peer-memory exchange (dist.cu): the slots were stored into this rank's window by its peers, each followed by the
    // peer's epoch flag; epoch = ctl[0] + 1, advanced by the last block of this kernel
    uint32_t epoch = 0;
    if (ctl) {
        epoch = *reinterpret_cast<volatile uint32_t*>(ctl) + 1;
        if (threadIdx.x < n_ranks) {
            const volatile uint32_t* f = slot_flag + threadIdx.x;
            const long long t0 = clock64();
            while ((int32_t)(*f - epoch) < 0) {
                __nanosleep(40);
                if (clock64() - t0 > 8000000000LL) __trap();       // a peer never arrived
            }
        }
        __threadfence_system();
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int acc = 0;
        for (int r = 0; r < n_ranks; r++) {
            prefix[r] = acc;
            int c = __ldcg(reinterpret_cast<const int*>(slots + (size_t)r * slot_records));
            acc += c < 0 ? 0 : (c < slot_records - 1 ? c : slot_records - 1);
        }
        prefix[n_ranks] = acc < n_cap ? acc : n_cap;
    }
    __syncthreads();
    const int n = prefix[n_ranks];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *n_out = n;
    float4 lf = make_float4(0.f, 0.f, 0.f, 0.f), rf = lf;
    if (i < n) {
        int r = 0;
        while (r + 1 < n_ranks && prefix[r + 1] <= i) r++;
        const int4 raw = __ldcg(reinterpret_cast<const int4*>(slots + (size_t)r * slot_records + 1 + (i - prefix[r])));
        erp_dmatch m;
        m.queryIdx = raw.x; m.trainIdx = raw.y; m.imgIdx = raw.z; m.distance = __int_as_float(raw.w);
        out[i] = m;
        double x, y, z;
        pixel_to_bearing(reinterpret_cast<const float*>(lxy + (size_t)m.queryIdx * stride), W, H, x, y, z);
        l3[3 * (size_t)i] = x; l3[3 * (size_t)i + 1] = y; l3[3 * (size_t)i + 2] = z;
        lf = make_float4((float)x, (float)y, (float)z, 0.f);
        l4[i] = lf;
        pixel_to_bearing(reinterpret_cast<const float*>(rxy + (size_t)m.trainIdx * stride), W, H, x, y, z);
        r3[3 * (size_t)i] = x; r3[3 * (size_t)i + 1] = y; r3[3 * (size_t)i + 2] = z;
        rf = make_float4((float)x, (float)y, (float)z, 0.f);
        r4[i] = rf;
    }
    if (Ks) prep_k_slot(i, n, lf, rf, Ks, w);
    if (ctl) {
        // every block has read the epoch and the slots: the last one to finish advances the epoch
        __syncthreads();
        if (threadIdx.x == 0) last = atomicAdd(ctl + 3, 1u) == gridDim.x - 1;
        __syncthreads();
        if (last && threadIdx.x == 0) { ctl[3] = 0; *reinterpret_cast<volatile uint32_t*>(ctl) = epoch; }
    }
}

// the same for keypoint pairs that are already gathered (erp_ransac_pixels): slot i of both views
__global__ void bearings_pair_kernel(const char* __restrict__ lxy, const char* __restrict__ rxy, size_t stride, int n, int W, int H,
                                     double* __restrict__ l3, double* __restrict__ r3, float4* __restrict__ l4, float4* __restrict__ r4,
                                     float* __restrict__ Ks, int32_t* __restrict__ w)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float4 lf = make_float4(0.f, 0.f, 0.f, 0.f), rf = lf;
    if (i < n) {
        double x, y, z;
        pixel_to_bearing(reinterpret_cast<const float*>(lxy + (size_t)i * stride), W, H, x, y, z);
        l3[3 * (size_t)i] = x; l3[3 * (size_t)i + 1] = y; l3[3 * (size_t)i + 2] = z;
        lf = make_float4((float)x, (float)y, (float)z, 0.f);
        l4[i] = lf;
        pixel_to_bearing(reinterpret_cast<const float*>(rxy + (size_t)i * stride), W, H, x, y, z);
        r3[3 * (size_t)i] = x; r3[3 * (size_t)i + 1] = y; r3[3 * (size_t)i + 2] = z;
        rf = make_float4((float)x, (float)y, (float)z, 0.f);
        r4[i] = rf;
    }
    if (Ks) prep_k_slot(i, n, lf, rf, Ks, w);
}

__global__ void pack4_kernel(const double* __restrict__ v3, int n, float4* __restrict__ v4)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v4[i] = make_float4((float)v3[3 * (size_t)i], (float)v3[3 * (size_t)i + 1], (float)v3[3 * (size_t)i + 2], 0.f);
}

// ------------------------------------------------------------------ Philox4x32-10 sampler
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}

// S distinct indices in [0,m): counter (hyp_lo, hyp_hi, block, 'ERP8'), key = seed; same spec as
// oracle/erp_oracle.c: orc_philox_samples.  out may be shared or global memory.
__device__ void philox_sample(uint64_t seed, uint64_t hyp, int m, int S, int32_t* out)
{
    int count = 0;
    uint32_t block = 0;
    while (count < S) {
        uint32_t c[4] = {(uint32_t)hyp, (uint32_t)(hyp >> 32), block++, 0x45525038u};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        for (int w = 0; w < 4 && count < S; w++) {
            int32_t idx = (int32_t)__umulhi(c[w], (uint32_t)m);
            bool dup = false;
            for (int j = 0; j < count; j++) dup |= out[j] == idx;
            if (!dup) out[count++] = idx;
        }
    }
}

__global__ void philox_table_kernel(uint64_t seed, uint64_t hyp0, int H, int S, int m, int32_t* table)
{
    int h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h < H) philox_sample(seed, hyp0 + h, m, S, table + (size_t)h * S);
}

// ------------------------------------------------------------------ Gram matrices G = A^T A
// upper-triangle index e -> (i,j), i <= j, row-major order
__constant__ uint8_t kTriI[45] = {0,0,0,0,0,0,0,0,0, 1,1,1,1,1,1,1,1, 2,2,2,2,2,2,2, 3,3,3,3,3,3, 4,4,4,4,4, 5,5,5,5, 6,6,6, 7,7, 8};
__constant__ uint8_t kTriJ[45] = {0,1,2,3,4,5,6,7,8, 1,2,3,4,5,6,7,8, 2,3,4,5,6,7,8, 3,4,5,6,7,8, 4,5,6,7,8, 5,6,7,8, 6,7,8, 7,8, 8};

constexpr int GW = 4;          // warps (hypotheses) per block in the small-sample kernel
constexpr int SMALL_S = 32;

// One warp per hypothesis, S <= 32 (the minimal-sample RANSAC case, S = 8).
// lane s builds row a_s = kron(l_s, r_s) (eight_point.cpp:28-36); lanes then own Gram entries.
__global__ void __launch_bounds__(GW * 32)
gram_small_kernel(const double* __restrict__ l3, const double* __restrict__ r3, int m_cap, const int32_t* __restrict__ m_dev,
                  const int32_t* __restrict__ samples, int H, int S, uint64_t seed, uint64_t hyp0,
                  const uint64_t* __restrict__ packed_dev, double* __restrict__ G /* H x 45 */)
{
    __shared__ double a[GW][SMALL_S][9];
    __shared__ int32_t smp[GW][SMALL_S];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int h = blockIdx.x * GW + w;
    if (h >= H) return;
    const int m = dev_len(m_dev, m_cap);
    if (m < S) {                                            // too few correspondences (device count): a zero system
        for (int e = lane; e < 45; e += 32) G[(size_t)h * 45 + e] = 0.0;
        return;
    }
    if (packed_dev) hyp0 = 0xFFFFFFFFull - (*packed_dev & 0xFFFFFFFFull);      // replay of the winner: its id is in the packed word
    if (samples) { if (lane < S) smp[w][lane] = samples[(size_t)h * S + lane]; }
    else if (lane == 0) philox_sample(seed, hyp0 + h, m, S, smp[w]);
    __syncwarp();
    if (lane < S) {
        int idx = smp[w][lane];
        double lx = l3[3 * (size_t)idx], ly = l3[3 * (size_t)idx + 1], lz = l3[3 * (size_t)idx + 2];
        double rx = r3[3 * (size_t)idx], ry = r3[3 * (size_t)idx + 1], rz = r3[3 * (size_t)idx + 2];
        double* o = a[w][lane];
        o[0] = lx * rx; o[1] = lx * ry; o[2] = lx * rz;
        o[3] = ly * rx; o[4] = ly * ry; o[5] = ly * rz;
        o[6] = lz * rx; o[7] = lz * ry; o[8] = lz * rz;
    }
    __syncwarp();
    for (int e = lane; e < 45; e += 32) {
        int i = kTriI[e], j = kTriJ[e];
        double acc = 0.0;
        for (int s = 0; s < S; s++) acc = __fma_rn(a[w][s][i], a[w][s][j], acc);
        G[(size_t)h * 45 + e] = acc;
    }
}

// One block per hypothesis for large samples (reference mode S = int(0.25 m), and the refit):
// every thread accumulates all 45 entries over a strided subset of rows, then a fixed-order
// tree reduction (deterministic).  index source: samples table, mask (compact on the fly), or all.
constexpr int GL_THREADS = 256;
__global__ void __launch_bounds__(GL_THREADS)
gram_large_kernel(const double* __restrict__ l3, const double* __restrict__ r3, int m,
                  const int32_t* __restrict__ samples, int S, const uint8_t* __restrict__ mask,
                  double* __restrict__ G /* gridDim.y x gridDim.x x 45 partials */)
{
    // blockIdx.y = hypothesis, blockIdx.x = slice of its rows
    const int h = blockIdx.y;
    double acc[45];
#pragma unroll
    for (int e = 0; e < 45; e++) acc[e] = 0.0;
    const int stride = gridDim.x * GL_THREADS;
    for (int s = blockIdx.x * GL_THREADS + threadIdx.x; s < S; s += stride) {
        int idx = samples ? samples[(size_t)h * S + s] : s;
        if (mask && !mask[idx]) continue;
        double v[9];
        {
            double lx = l3[3 * (size_t)idx], ly = l3[3 * (size_t)idx + 1], lz = l3[3 * (size_t)idx + 2];
            double rx = r3[3 * (size_t)idx], ry = r3[3 * (size_t)idx + 1], rz = r3[3 * (size_t)idx + 2];
            v[0] = lx * rx; v[1] = lx * ry; v[2] = lx * rz;
            v[3] = ly * rx; v[4] = ly * ry; v[5] = ly * rz;
            v[6] = lz * rx; v[7] = lz * ry; v[8] = lz * rz;
        }
        int e = 0;
#pragma unroll
        for (int i = 0; i < 9; i++)
#pragma unroll
            for (int j = i; j < 9; j++) { acc[e] = __fma_rn(v[i], v[j], acc[e]); e++; }
    }
    __shared__ double red[GL_THREADS / 32][45];
#pragma unroll
    for (int e = 0; e < 45; e++) {
        double x = acc[e];
        for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][e] = x;
    }
    __syncthreads();
    if (threadIdx.x < 45) {
        double x = 0.0;
        for (int w = 0; w < GL_THREADS / 32; w++) x += red[w][threadIdx.x];
        G[((size_t)h * gridDim.x + blockIdx.x) * 45 + threadIdx.x] = x;
    }
}

// sum the per-slice partials in slice order: G[h] = sum_b P[h][b]
__global__ void gram_finish_kernel(const double* __restrict__ P, int H, int slices, double* __restrict__ G)
{
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= H * 45) return;
    int h = i / 45, e = i % 45;
    double x = 0.0;
    for (int b = 0; b < slices; b++) x += P[((size_t)h * slices + b) * 45 + e];
    G[i] = x;
}

// ------------------------------------------------------------------ 3x3 helpers
struct M3 { double v[9]; };

__device__ __forceinline__ M3 mul3(const M3& A, const M3& B)
{
    M3 C;
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++)
            C.v[3 * i + j] = A.v[3 * i] * B.v[j] + A.v[3 * i + 1] * B.v[3 + j] + A.v[3 * i + 2] * B.v[6 + j];
    return C;
}

__device__ __forceinline__ double det3(const M3& M)
{
    return M.v[0] * (M.v[4] * M.v[8] - M.v[5] * M.v[7]) - M.v[1] * (M.v[3] * M.v[8] - M.v[5] * M.v[6]) +
           M.v[2] * (M.v[3] * M.v[7] - M.v[4] * M.v[6]);
}

// OpenCV's Jacobi rotation coefficients for the pair with squared norms a, b and dot p
__device__ __forceinline__ void cv_rotation(double a, double b, double p, double& c, double& s)
{
    p *= 2;
    double beta = a - b, gamma = hypot(p, beta);
    if (beta < 0) {
        double delta = (gamma - beta) * 0.5;
        s = sqrt(delta / gamma);
        c = p / (gamma * s * 2);
    } else {
        c = sqrt((gamma + beta) / (gamma * 2));
        s = p / (gamma * c * 2);
    }
}

// cv::SVD::compute on a 3x3 (m == n): one-sided Jacobi on the columns of E.
// U = normalised rotated columns, Vt rows = right singular vectors, w descending.
__device__ void svd3(const M3& E, double w[3], M3& U, M3& Vt)
{
    const double eps = DBL_EPSILON * 10;
    double At[3][3], V[3][3], W[3];   // At rows = columns of E
#pragma unroll
    for (int i = 0; i < 3; i++) {
#pragma unroll
        for (int k = 0; k < 3; k++) { At[i][k] = E.v[3 * k + i]; V[i][k] = (i == k) ? 1.0 : 0.0; }
        W[i] = At[i][0] * At[i][0] + At[i][1] * At[i][1] + At[i][2] * At[i][2];
    }
    for (int iter = 0; iter < 30; iter++) {
        bool changed = false;
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
            for (int j = i + 1; j < 3; j++) {
                double a = W[i], b = W[j];
                double p = At[i][0] * At[j][0] + At[i][1] * At[j][1] + At[i][2] * At[j][2];
                if (fabs(p) <= eps * sqrt(a * b)) continue;
                double c, s;
                cv_rotation(a, b, p, c, s);
                a = b = 0;
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    double t0 = c * At[i][k] + s * At[j][k], t1 = -s * At[i][k] + c * At[j][k];
                    At[i][k] = t0; At[j][k] = t1;
                    a += t0 * t0; b += t1 * t1;
                    double v0 = c * V[i][k] + s * V[j][k], v1 = -s * V[i][k] + c * V[j][k];
                    V[i][k] = v0; V[j][k] = v1;
                }
                W[i] = a; W[j] = b;
                changed = true;
            }
        if (!changed) break;
    }
#pragma unroll
    for (int i = 0; i < 3; i++) W[i] = sqrt(At[i][0] * At[i][0] + At[i][1] * At[i][1] + At[i][2] * At[i][2]);
    // selection sort, descending, strict < as OpenCV
#pragma unroll
    for (int i = 0; i < 2; i++) {
        int j = i;
#pragma unroll
        for (int k = i + 1; k < 3; k++) if (W[j] < W[k]) j = k;
        if (i != j) {
            double t = W[i]; W[i] = W[j]; W[j] = t;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                t = At[i][k]; At[i][k] = At[j][k]; At[j][k] = t;
                t = V[i][k]; V[i][k] = V[j][k]; V[j][k] = t;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 3; i++) {
        w[i] = W[i];
        // OpenCV substitutes a pseudo-random orthogonal vector when W <= DBL_MIN; an exactly
        // singular E has no usable third column, so the device leaves it zero and lets
        // decompose() rebuild it from the other two.
        double s = W[i] > DBL_MIN ? 1.0 / W[i] : 0.0;
#pragma unroll
        for (int k = 0; k < 3; k++) { U.v[3 * k + i] = At[i][k] * s; Vt.v[3 * i + k] = V[i][k]; }
    }
}

// erp_rotation.cpp:43-63
__device__ __forceinline__ void rot2eular(const M3& R, double e[3])
{
    double sy = sqrt(R.v[8] * R.v[8] + R.v[5] * R.v[5]);
    e[0] = sy < 1e-6 ? 0.0 : atan2(-R.v[5], R.v[8]);
    e[1] = atan2(R.v[2], sy);
    e[2] = atan2(-R.v[1], R.v[0]);
}

__device__ __forceinline__ float max_vec3(float a, float b, float c)   // eight_point.cpp:6-14
{
    if ((a > b) && (a > c)) return a;
    else if (b > c) return b;
    else return c;
}

// cv::decomposeEssentialMat + rot2eular + validity (eight_point.cpp:53-84)
__device__ void decompose_pose(const M3& Ec, float* pose)
{
    double D[3];
    M3 U, Vt;
    svd3(Ec, D, U, Vt);
    if (!(D[2] > DBL_MIN)) {   // exactly rank-2 input: third left vector = u1 x u2
        U.v[2] = U.v[3] * U.v[7] - U.v[6] * U.v[4];
        U.v[5] = U.v[6] * U.v[1] - U.v[0] * U.v[7];
        U.v[8] = U.v[0] * U.v[4] - U.v[3] * U.v[1];
    }
    if (det3(U) < 0) for (int i = 0; i < 9; i++) U.v[i] = -U.v[i];
    if (det3(Vt) < 0) for (int i = 0; i < 9; i++) Vt.v[i] = -Vt.v[i];
    M3 Wm = {{0, 1, 0, -1, 0, 0, 0, 0, 1}}, Wt = {{0, -1, 0, 1, 0, 0, 0, 0, 1}};
    M3 R1 = mul3(mul3(U, Wm), Vt), R2 = mul3(mul3(U, Wt), Vt);
    double e1[3], e2[3];
    rot2eular(R1, e1);
    rot2eular(R2, e2);
    float f1[3] = {(float)e1[0], (float)e1[1], (float)e1[2]};
    float f2[3] = {(float)e2[0], (float)e2[1], (float)e2[2]};
    pose[0] = f1[0]; pose[1] = f1[1]; pose[2] = f1[2];
    pose[3] = f2[0]; pose[4] = f2[1]; pose[5] = f2[2];
    pose[6] = (float)U.v[2]; pose[7] = (float)U.v[5]; pose[8] = (float)U.v[8];
    pose[9] = ((double)max_vec3(fabsf(f1[0]), fabsf(f1[1]), fabsf(f1[2])) < 1.57) ? 1.f : 0.f;
    pose[10] = ((double)max_vec3(fabsf(f2[0]), fabsf(f2[1]), fabsf(f2[2])) < 1.57) ? 1.f : 0.f;
    pose[11] = 0.f;
}

// rank-2 projection (eight_point.cpp:45-50: SVD, sigma3 <- 0, recompose), optional pose.
// U diag(s1, s2, 0) V^T = E - (E v3) v3^T with v3 the right singular vector of the smallest singular value, i.e. the
// eigenvector of M = E^T E for its smallest eigenvalue.  A full one-sided Jacobi SVD (hypot, sqrt and two divisions per
// rotation, ~15 rotations) was 40 % of the minimal-sample solver; here the eigenvalue comes from Newton's iteration on
// the characteristic cubic started at 0 (monotone from below: the cubic is increasing and concave up to its first
// root) and v3 from the largest cross product of two rows of M - lambda I: ~150 flops, one square root.  The result is
// the same matrix to working precision; a (numerically) double smallest singular value falls back to the SVD.  Next to a
// double root Newton converges only linearly (each step halves the distance), so a loop that ends at its cap with steps
// still above their rounding noise has not found lambda3 (sigma3 close to sigma2) and falls back as well.
__device__ __forceinline__ bool rank2_project_fast(const M3& E, M3& Ec)
{
    double m[6];                                  // M = E^T E, upper triangle: 00 01 02 11 12 22
    m[0] = E.v[0] * E.v[0] + E.v[3] * E.v[3] + E.v[6] * E.v[6];
    m[1] = E.v[0] * E.v[1] + E.v[3] * E.v[4] + E.v[6] * E.v[7];
    m[2] = E.v[0] * E.v[2] + E.v[3] * E.v[5] + E.v[6] * E.v[8];
    m[3] = E.v[1] * E.v[1] + E.v[4] * E.v[4] + E.v[7] * E.v[7];
    m[4] = E.v[1] * E.v[2] + E.v[4] * E.v[5] + E.v[7] * E.v[8];
    m[5] = E.v[2] * E.v[2] + E.v[5] * E.v[5] + E.v[8] * E.v[8];
    const double tr = m[0] + m[3] + m[5];
    if (!(tr > 0.0) || !(tr < INFINITY)) return false;
    // f(x) = x^3 - c2 x^2 + c1 x - c0, roots = eigenvalues
    const double c2 = tr;
    const double c1 = (m[0] * m[3] - m[1] * m[1]) + (m[0] * m[5] - m[2] * m[2]) + (m[3] * m[5] - m[4] * m[4]);
    const double dE = det3(E), c0 = dE * dE;
    double x = 0.0, step = INFINITY, df = 0.0;
    for (int it = 0; it < 12; it++) {
        const double f = ((x - c2) * x + c1) * x - c0;
        df = (3.0 * x - 2.0 * c2) * x + c1;
        if (!(df > 0.0)) return false;            // the two smallest eigenvalues (nearly) coincide
        step = f / df;
        x -= step;
        if (fabs(step) <= 1e-17 * tr) break;
    }
    // at the cap: converged only if the last step was at the rounding noise of f / df (the Horner terms of f round to a
    // few ulp each), where the steps of a found root stall; a larger step is the linear approach to a double root
    if (!(fabs(step) <= 1e-17 * tr)) {
        const double ax = fabs(x);
        if (!(fabs(step) <= 16.0 * DBL_EPSILON * (((ax + c2) * ax + c1) * ax + c0) / df)) return false;
    }
    if (!(x >= 0.0)) x = 0.0;
    // rows of A = M - x I
    const double a00 = m[0] - x, a11 = m[3] - x, a22 = m[5] - x;
    const double r0[3] = {a00, m[1], m[2]}, r1[3] = {m[1], a11, m[4]}, r2[3] = {m[2], m[4], a22};
    double c[3][3];
    c[0][0] = r0[1] * r1[2] - r0[2] * r1[1]; c[0][1] = r0[2] * r1[0] - r0[0] * r1[2]; c[0][2] = r0[0] * r1[1] - r0[1] * r1[0];
    c[1][0] = r0[1] * r2[2] - r0[2] * r2[1]; c[1][1] = r0[2] * r2[0] - r0[0] * r2[2]; c[1][2] = r0[0] * r2[1] - r0[1] * r2[0];
    c[2][0] = r1[1] * r2[2] - r1[2] * r2[1]; c[2][1] = r1[2] * r2[0] - r1[0] * r2[2]; c[2][2] = r1[0] * r2[1] - r1[1] * r2[0];
    double n[3];
#pragma unroll
    for (int k = 0; k < 3; k++) n[k] = c[k][0] * c[k][0] + c[k][1] * c[k][1] + c[k][2] * c[k][2];
    const int best = n[0] >= n[1] ? (n[0] >= n[2] ? 0 : 2) : (n[1] >= n[2] ? 1 : 2);
    const double nb = best == 0 ? n[0] : (best == 1 ? n[1] : n[2]);
    // |r_i x r_j| ~ (l1 - l3)(l2 - l3): a tiny value means the smallest eigenvalue is not isolated
    if (!(nb > 1e-12 * tr * tr * tr * tr)) return false;
    const double inv = 1.0 / sqrt(nb);
    double v[3];
#pragma unroll
    for (int k = 0; k < 3; k++) v[k] = (best == 0 ? c[0][k] : (best == 1 ? c[1][k] : c[2][k])) * inv;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const double w = E.v[3 * i] * v[0] + E.v[3 * i + 1] * v[1] + E.v[3 * i + 2] * v[2];
#pragma unroll
        for (int j = 0; j < 3; j++) Ec.v[3 * i + j] = E.v[3 * i + j] - w * v[j];
    }
    return true;
}

template <bool WANT_POSE>
__device__ __forceinline__ void finish_hypothesis(const M3& E, double* __restrict__ Eout, float* __restrict__ pose)
{
    M3 Ec;
    if (!rank2_project_fast(E, Ec)) {
        double w[3];
        M3 U, Vt;
        svd3(E, w, U, Vt);
        M3 UD;
#pragma unroll
        for (int i = 0; i < 3; i++) { UD.v[3 * i] = U.v[3 * i] * w[0]; UD.v[3 * i + 1] = U.v[3 * i + 1] * w[1]; UD.v[3 * i + 2] = 0.0; }
        Ec = mul3(UD, Vt);
    }
#pragma unroll
    for (int k = 0; k < 9; k++) Eout[k] = Ec.v[k];
    if (WANT_POSE) decompose_pose(Ec, pose);
}

// ------------------------------------------------------------------ 9x9 Jacobi, thread per hypothesis
constexpr int SOLVE_THREADS = 64;
// symmetric index into the packed upper triangle
__host__ __device__ constexpr int tri(int i, int j) { return i <= j ? i * 9 - i * (i - 1) / 2 + (j - i) : j * 9 - j * (j - 1) / 2 + (i - j); }

template <bool WANT_POSE>
__global__ void __launch_bounds__(SOLVE_THREADS)
solve_kernel(const double* __restrict__ Gin, int H, int max_sweeps,
             double* __restrict__ Eout /* H x 9 */, float* __restrict__ pose /* H x 12 */)
{
    // V (rows = right singular vectors, OpenCV's Vt) lives in shared memory, element-major so
    // that the 64 threads of a block hit 64 consecutive doubles; G (45 doubles) in registers.
    __shared__ double Vs[81][SOLVE_THREADS];
    const int tid = threadIdx.x;
    const int h = blockIdx.x * SOLVE_THREADS + tid;
    if (h >= H) return;
    double G[45];
#pragma unroll
    for (int e = 0; e < 45; e++) G[e] = Gin[(size_t)h * 45 + e];
#pragma unroll
    for (int i = 0; i < 9; i++)
#pragma unroll
        for (int k = 0; k < 9; k++) Vs[i * 9 + k][tid] = (i == k) ? 1.0 : 0.0;

    const double eps = DBL_EPSILON * 10;
    for (int sweep = 0; sweep < max_sweeps; sweep++) {
        bool changed = false;
#pragma unroll
        for (int i = 0; i < 8; i++) {
#pragma unroll
            for (int j = i + 1; j < 9; j++) {
                double a = G[tri(i, i)], b = G[tri(j, j)], p = G[tri(i, j)];
                double ab = fmax(a, 0.0) * fmax(b, 0.0);
                // OpenCV's relative test, plus the floor a Gram matrix can resolve
                if (fabs(p) <= eps * sqrt(ab) || fabs(p) <= DBL_EPSILON * fmax(fabs(a), fabs(b))) continue;
                double c, s;
                cv_rotation(a, b, p, c, s);
                // G <- J^T G J  with  col_i' = c col_i + s col_j,  col_j' = -s col_i + c col_j
#pragma unroll
                for (int k = 0; k < 9; k++) {
                    if (k == i || k == j) continue;
                    double gi = G[tri(k, i)], gj = G[tri(k, j)];
                    G[tri(k, i)] = c * gi + s * gj;
                    G[tri(k, j)] = -s * gi + c * gj;
                }
                double cc = c * c, ss = s * s, cs = c * s;
                G[tri(i, i)] = cc * a + 2 * cs * p + ss * b;
                G[tri(j, j)] = ss * a - 2 * cs * p + cc * b;
                G[tri(i, j)] = (cc - ss) * p + cs * (b - a);
#pragma unroll
                for (int k = 0; k < 9; k++) {
                    double vi = Vs[i * 9 + k][tid], vj = Vs[j * 9 + k][tid];
                    Vs[i * 9 + k][tid] = c * vi + s * vj;
                    Vs[j * 9 + k][tid] = -s * vi + c * vj;
                }
                changed = true;
            }
        }
        if (!changed) break;
        // a Gram matrix cannot resolve off-diagonals below ~eps * trace: once they are all there, further
        // sweeps only churn rounding noise (the pairwise relative test above then never fires)
        double off = 0.0, trc = 0.0;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            trc += fabs(G[tri(i, i)]);
#pragma unroll
            for (int j = i + 1; j < 9; j++) off = __fma_rn(G[tri(i, j)], G[tri(i, j)], off);
        }
        if (off <= (64.0 * DBL_EPSILON * trc) * (64.0 * DBL_EPSILON * trc)) break;
    }
    // singular values = sqrt of the diagonal; OpenCV's descending selection sort decides which
    // row ends up last (vt.row(vt.rows-1), eight_point.cpp:42)
    double W[9];
    int perm[9];
#pragma unroll
    for (int i = 0; i < 9; i++) { W[i] = sqrt(fmax(G[tri(i, i)], 0.0)); perm[i] = i; }
    for (int i = 0; i < 8; i++) {
        int j = i;
        for (int k = i + 1; k < 9; k++) if (W[j] < W[k]) j = k;
        if (i != j) { double t = W[i]; W[i] = W[j]; W[j] = t; int q = perm[i]; perm[i] = perm[j]; perm[j] = q; }
    }
    const int last = perm[8];
    M3 E;
#pragma unroll
    for (int k = 0; k < 9; k++) E.v[k] = Vs[last * 9 + k][tid];

    finish_hypothesis<WANT_POSE>(E, Eout + (size_t)h * 9, pose ? pose + (size_t)h * ERP_POSE_FLOATS : nullptr);
}

// ------------------------------------------------------------------ minimal sample (S = 8), thread per hypothesis
// The 8 x 9 matrix A has a one-dimensional null space: e is the last column of Q in the QR
// factorisation of A^T (9 x 8), i.e. e = H0 H1 ... H7 e8 with the eight Householder reflectors that
// triangularise the columns kron(l_i, r_i).  About 500 fp64 FMAs instead of a 9 x 9 Jacobi eigen
// solve (~50k), working on A itself (condition number not squared), fully unrolled in registers.
// The sign of e is arbitrary (as in any SVD); everything downstream is sign invariant.
constexpr int MIN8_THREADS = 128;
template <bool WANT_POSE>
__global__ void __launch_bounds__(MIN8_THREADS)
min8_kernel(const double* __restrict__ l3, const double* __restrict__ r3, int m_cap, const int32_t* __restrict__ m_dev,
            const int32_t* __restrict__ samples, int H, uint64_t seed, uint64_t hyp0, const uint64_t* __restrict__ packed_dev,
            double* __restrict__ Eout, float* __restrict__ pose, const Min8Fused fused)
{
    const int h = blockIdx.x * MIN8_THREADS + threadIdx.x;
    // fused tail of the RANSAC chain: the hypothesis operand of the tensor-core search, its cleared bounds and pass A's shape
    if (fused.Es && h == 0) { fused.w[W_DYN_A] = H; fused.w[W_DYN_A + 1] = 0; fused.w[W_DYN_A + 2] = fused.w[W_N0]; fused.w[W_DYN_A + 3] = fused.w[W_M]; }
    if (h >= H) return;
    const int m = dev_len(m_dev, m_cap);
    if (packed_dev) hyp0 = 0xFFFFFFFFull - (*packed_dev & 0xFFFFFFFFull);      // replay of the winner: its id is in the packed word
    if (m < 8) {                                            // too few correspondences (device count): the zero matrix
#pragma unroll
        for (int k = 0; k < 9; k++) Eout[(size_t)h * 9 + k] = 0.0;
        if (fused.Es) { zero_row(fused.Es + (size_t)h * 32); fused.upper[h] = 0; fused.upper[(size_t)H + h] = 0; }
        return;
    }
    int32_t idx[8];
    if (samples) {
#pragma unroll
        for (int j = 0; j < 8; j++) idx[j] = samples[(size_t)h * 8 + j];
    } else philox_sample(seed, hyp0 + h, m, 8, idx);

    double M[8][9];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const size_t o = 3 * (size_t)idx[j];
        double lx = l3[o], ly = l3[o + 1], lz = l3[o + 2];
        double rx = r3[o], ry = r3[o + 1], rz = r3[o + 2];
        M[j][0] = lx * rx; M[j][1] = lx * ry; M[j][2] = lx * rz;
        M[j][3] = ly * rx; M[j][4] = ly * ry; M[j][5] = ly * rz;
        M[j][6] = lz * rx; M[j][7] = lz * ry; M[j][8] = lz * rz;
    }
    double beta[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        double tail2 = 0.0;
#pragma unroll
        for (int k = j + 1; k < 9; k++) tail2 = __fma_rn(M[j][k], M[j][k], tail2);
        const double x0 = M[j][j];
        const double nrm = sqrt(__fma_rn(x0, x0, tail2));
        const double v0 = x0 >= 0.0 ? x0 + nrm : x0 - nrm;      // x0 - alpha, alpha = -sign(x0) |x|
        M[j][j] = v0;
        const double vtv = __fma_rn(v0, v0, tail2);
        beta[j] = vtv > 0.0 ? 2.0 / vtv : 0.0;
#pragma unroll
        for (int c = j + 1; c < 8; c++) {
            double d = 0.0;
#pragma unroll
            for (int k = j; k < 9; k++) d = __fma_rn(M[j][k], M[c][k], d);
            d *= beta[j];
#pragma unroll
            for (int k = j; k < 9; k++) M[c][k] = __fma_rn(-d, M[j][k], M[c][k]);
        }
    }
    double q[9] = {0, 0, 0, 0, 0, 0, 0, 0, 1};
#pragma unroll
    for (int j = 7; j >= 0; j--) {
        double d = 0.0;
#pragma unroll
        for (int k = j; k < 9; k++) d = __fma_rn(M[j][k], q[k], d);
        d *= beta[j];
#pragma unroll
        for (int k = j; k < 9; k++) q[k] = __fma_rn(-d, M[j][k], q[k]);
    }
    double n2 = 0.0;
#pragma unroll
    for (int k = 0; k < 9; k++) n2 = __fma_rn(q[k], q[k], n2);
    const double inv = n2 > 0.0 ? 1.0 / sqrt(n2) : 0.0;
    M3 E;
#pragma unroll
    for (int k = 0; k < 9; k++) E.v[k] = q[k] * inv;
    finish_hypothesis<WANT_POSE>(E, Eout + (size_t)h * 9, pose ? pose + (size_t)h * ERP_POSE_FLOATS : nullptr);
    if (fused.Es) {
        float e[9];
        scale_E(Eout + (size_t)h * 9, e);
        RowScale rs;
        rs.metric = fused.metric; rs.tau = fused.tau; rs.sin_tau = fused.sin_tau;
        write_e_row(e, fused.big, fused.Es + (size_t)h * 32, row_gain(e, rs, fused.w));
        fused.upper[h] = 0; fused.upper[(size_t)H + h] = 0;
    }
}

// ------------------------------------------------------------------ one 9x9 solve on one warp
// solve_kernel keeps a whole problem in one thread (right for a million hypotheses, 0.3 ms of serial
// latency for a single refit).  Here lane k owns row/column k of G and column k of V in shared memory
// and every rotation is applied by nine lanes at once; same pivot order and element formulas as
// solve_kernel, so the two agree to the last bit.
struct Solve1Smem { double G[9][9], V[9][9]; int flag[1]; };

// one warp (lane k); Gin: the packed upper triangle in global or shared memory
template <bool WANT_POSE>
__device__ void solve1_warp(Solve1Smem& sm, const double* Gin, int max_sweeps, double* __restrict__ Eout, float* __restrict__ pose)
{
    double (&G)[9][9] = sm.G;
    double (&V)[9][9] = sm.V;
    int (&flag)[1] = sm.flag;
    const int k = threadIdx.x & 31;
    if (k < 9)
        for (int j = 0; j < 9; j++) { G[k][j] = Gin[tri(k, j)]; V[k][j] = (k == j) ? 1.0 : 0.0; }
    __syncwarp();
    const double eps = DBL_EPSILON * 10;
    for (int sweep = 0; sweep < max_sweeps; sweep++) {
        if (k == 0) flag[0] = 0;
        __syncwarp();
        for (int i = 0; i < 8; i++) {
            for (int j = i + 1; j < 9; j++) {
                const double a = G[i][i], b = G[j][j], p = G[i][j];
                const double ab = fmax(a, 0.0) * fmax(b, 0.0);
                const bool skip = fabs(p) <= eps * sqrt(ab) || fabs(p) <= DBL_EPSILON * fmax(fabs(a), fabs(b));   // warp-uniform
                if (skip) continue;
                double c, s;
                cv_rotation(a, b, p, c, s);
                __syncwarp();
                if (k < 9) {
                    if (k != i && k != j) {
                        const double gi = G[k][i], gj = G[k][j];
                        const double ni = c * gi + s * gj, nj = -s * gi + c * gj;
                        G[k][i] = ni; G[i][k] = ni; G[k][j] = nj; G[j][k] = nj;
                    }
                    const double vi = V[i][k], vj = V[j][k];
                    V[i][k] = c * vi + s * vj;
                    V[j][k] = -s * vi + c * vj;
                }
                if (k == 0) {
                    const double cc = c * c, ss = s * s, sc = c * s;
                    G[i][i] = cc * a + 2 * sc * p + ss * b;
                    G[j][j] = ss * a - 2 * sc * p + cc * b;
                    const double nij = (cc - ss) * p + sc * (b - a);
                    G[i][j] = nij; G[j][i] = nij;
                    flag[0] = 1;
                }
                __syncwarp();
            }
        }
        __syncwarp();
        if (!flag[0]) break;
        double off = 0.0, trc = 0.0;
        for (int i = 0; i < 9; i++) {
            trc += fabs(G[i][i]);
            for (int j = i + 1; j < 9; j++) off = __fma_rn(G[i][j], G[i][j], off);
        }
        if (off <= (64.0 * DBL_EPSILON * trc) * (64.0 * DBL_EPSILON * trc)) break;
    }
    if (k != 0) return;
    double W[9];
    int perm[9];
    for (int i = 0; i < 9; i++) { W[i] = sqrt(fmax(G[i][i], 0.0)); perm[i] = i; }
    for (int i = 0; i < 8; i++) {
        int j = i;
        for (int q = i + 1; q < 9; q++) if (W[j] < W[q]) j = q;
        if (i != j) { double t = W[i]; W[i] = W[j]; W[j] = t; int q = perm[i]; perm[i] = perm[j]; perm[j] = q; }
    }
    M3 E;
    for (int q = 0; q < 9; q++) E.v[q] = V[perm[8]][q];
    finish_hypothesis<WANT_POSE>(E, Eout, pose);
}

template <bool WANT_POSE>
__global__ void __launch_bounds__(32)
solve1_kernel(const double* __restrict__ Gin, int max_sweeps, double* __restrict__ Eout, float* __restrict__ pose)
{
    __shared__ Solve1Smem sm;
    solve1_warp<WANT_POSE>(sm, Gin, max_sweeps, Eout, pose);
}

// ------------------------------------------------------------------ refit solve: smallest eigenvector by inverse iteration
// The refit of a RANSAC call is the right singular vector of the smallest singular value of the inlier matrix A
// (eight_point.cpp:38-43), i.e. the eigenvector of the smallest eigenvalue of G = A^T A (9 x 9, SPD).  A Jacobi eigen
// solve on one warp is a serial chain of ~300 rotations (130 us measured, most of the fixed cost of a call).  The
// winning minimal-sample model is already close to that vector, and the smallest eigenvalue (noise) is orders of
// magnitude below the next one (signal), so inverse iteration  x <- normalise((G + mu I)^-1 x)  from x0 = E_best gains
// several digits per step: one 9 x 9 Cholesky factorisation and a handful of triangular solves on one thread, ~5 us.
// mu = 1e-12 trace(G) keeps the factorisation defined for noise-free input (an exactly singular G).  The sign follows
// E_best.  Only used for the RANSAC refit (sign-invariant consumers); the reference-mode solves keep OpenCV's Jacobi.
// The iteration stops when an iterate changes by less than 1e-14, or when the change stops halving and x is an
// eigenvector to the rounding floor of G: ||G x - (x^T G x) x|| <= 64 eps trace(G), the floor the Jacobi solves stop at
// too (the error of x is then at most that residual over the gap lambda2 - lambda1).  Each step shrinks the error only
// by (lambda1 + mu) / (lambda2 + mu): on a low-parallax pair, where the two smallest eigenvalues are both noise and
// within a factor of a few, the change stops halving long before the floor and the cap may come first.  It then returns
// false without writing anything, and the caller solves the same G with the one-warp Jacobi.
__device__ bool refit_inverse_iteration(const double* Gp /* packed upper triangle */, const double* x0, double* __restrict__ Eout,
                                        float* __restrict__ pose)
{
    double L[9][9];
    double trace = 0.0;
#pragma unroll
    for (int i = 0; i < 9; i++) trace += Gp[tri(i, i)];
    const double mu = 1e-12 * trace + 1e-300;
    double inv[9];
#pragma unroll
    for (int j = 0; j < 9; j++) {
        double d = Gp[tri(j, j)] + mu;
#pragma unroll
        for (int k = 0; k < j; k++) d = __fma_rn(-L[j][k], L[j][k], d);
        d = d > mu * 1e-3 ? d : mu * 1e-3;                    // numerically semi-definite: keep the factor finite
        const double r = sqrt(d);
        L[j][j] = r;
        inv[j] = 1.0 / r;
#pragma unroll
        for (int i = j + 1; i < 9; i++) {
            double v = Gp[tri(j, i)];
#pragma unroll
            for (int k = 0; k < j; k++) v = __fma_rn(-L[i][k], L[j][k], v);
            L[i][j] = v * inv[j];
        }
    }
    double x[9], n2 = 0.0;
#pragma unroll
    for (int i = 0; i < 9; i++) { x[i] = x0[i]; n2 = __fma_rn(x[i], x[i], n2); }
    if (!(n2 > 0.0)) { x[8] = 1.0; n2 = 1.0; }
    {
        const double s = 1.0 / sqrt(n2);
#pragma unroll
        for (int i = 0; i < 9; i++) x[i] *= s;
    }
    const double floor2 = (64.0 * DBL_EPSILON * trace) * (64.0 * DBL_EPSILON * trace);
    double prev = INFINITY;
    bool converged = false;
    for (int it = 0; it < 24; it++) {
        double y[9];
#pragma unroll
        for (int i = 0; i < 9; i++) {                        // L z = x
            double v = x[i];
#pragma unroll
            for (int k = 0; k < i; k++) v = __fma_rn(-L[i][k], y[k], v);
            y[i] = v * inv[i];
        }
#pragma unroll
        for (int i = 8; i >= 0; i--) {                       // L^T y = z
            double v = y[i];
#pragma unroll
            for (int k = i + 1; k < 9; k++) v = __fma_rn(-L[k][i], y[k], v);
            y[i] = v * inv[i];
        }
        double yy = 0.0, xy = 0.0;
#pragma unroll
        for (int i = 0; i < 9; i++) { yy = __fma_rn(y[i], y[i], yy); xy = __fma_rn(x[i], y[i], xy); }
        if (!(yy > 0.0) || !(yy < INFINITY)) break;
        const double s = (xy < 0.0 ? -1.0 : 1.0) / sqrt(yy);
        double diff = 0.0;
#pragma unroll
        for (int i = 0; i < 9; i++) { const double v = y[i] * s; diff = fmax(diff, fabs(v - x[i])); x[i] = v; }
        // a change below 1e-14 leaves an error of at most 1e-14 r / (1 - r), r = lambda1 / lambda2, which is below the
        // floor 64 eps trace / (lambda2 - lambda1) for every r
        if (diff < 1e-14) { converged = true; break; }
        const bool stalled = it > 0 && diff >= 0.5 * prev;
        prev = diff;
        // the change no longer halves: at the rounding floor of the solves, or lambda1 / lambda2 >= 1/2 and still far
        // from it; the residual tells the two apart (also at the cap)
        if (!stalled && it < 23) continue;
        double gx[9], rho = 0.0;
#pragma unroll
        for (int i = 0; i < 9; i++) {
            double v = 0.0;
#pragma unroll
            for (int k = 0; k < 9; k++) v = __fma_rn(Gp[tri(i, k)], x[k], v);
            gx[i] = v;
            rho = __fma_rn(x[i], v, rho);
        }
        double res2 = 0.0;
#pragma unroll
        for (int i = 0; i < 9; i++) { const double d = __fma_rn(-rho, x[i], gx[i]); res2 = __fma_rn(d, d, res2); }
        if (res2 <= floor2) { converged = true; break; }
    }
    if (!converged) return false;
    M3 E;
#pragma unroll
    for (int k = 0; k < 9; k++) E.v[k] = x[k];
    finish_hypothesis<true>(E, Eout, pose);
    return true;
}

// ------------------------------------------------------------------ end of a RANSAC call, one launch
// Inlier mask of the winning model, the Gram matrix of its inliers and the least-squares refit (eight_point.cpp:16-50 on
// the inlier set): every block marks 256 correspondences and reduces their 45 Gram entries in a fixed order; the last
// block to finish (one ticket) sums the per-block partials in block order (deterministic), solves the 9 x 9 system on its
// first warp (inverse iteration on lane 0; the one-warp Jacobi when that does not converge) and writes the whole
// erp_ransac_result.  cnt: [0] inliers, [1] ticket (both zeroed by the caller).
constexpr int FIN_THREADS = 256;
template <int METRIC>
__global__ void __launch_bounds__(FIN_THREADS)
finish_kernel(const double* __restrict__ Eb, const uint64_t* __restrict__ packed_dev, const double* __restrict__ l3,
              const double* __restrict__ r3, const float4* __restrict__ l4, const float4* __restrict__ r4, int m_cap,
              const int32_t* __restrict__ m_dev, float tau, float tau2, float sin2, uint8_t* __restrict__ mask,
              double* __restrict__ P /* gridDim.x x 45 */, int32_t* __restrict__ cnt, erp_ransac_result* __restrict__ out)
{
    __shared__ float Es[9];
    __shared__ double red[FIN_THREADS / 32][45];
    __shared__ double Gs[45];
    __shared__ Solve1Smem s1;
    __shared__ int last, jacobi;
    const int m = dev_len(m_dev, m_cap);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) scale_E(Eb, Es);
    __syncthreads();
    const int c = blockIdx.x * FIN_THREADS + threadIdx.x;
    bool in = false;
    double v[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (c < m) {
        float e[9];
#pragma unroll
        for (int i = 0; i < 9; i++) e[i] = Es[i];
        const float4 l = l4[c], r = r4[c];
        float k[9];
        kron9(l, r, k);
        in = inlier<METRIC>(e, k, l, r, tau, tau2, sin2);
        if (mask) mask[c] = in ? 1 : 0;
        if (in) {
            const double lx = l3[3 * (size_t)c], ly = l3[3 * (size_t)c + 1], lz = l3[3 * (size_t)c + 2];
            const double rx = r3[3 * (size_t)c], ry = r3[3 * (size_t)c + 1], rz = r3[3 * (size_t)c + 2];
            v[0] = lx * rx; v[1] = lx * ry; v[2] = lx * rz;
            v[3] = ly * rx; v[4] = ly * ry; v[5] = ly * rz;
            v[6] = lz * rx; v[7] = lz * ry; v[8] = lz * rz;
        }
    }
    const int n_in = __reduce_add_sync(0xffffffffu, in ? 1 : 0);
    if (lane == 0 && n_in) atomicAdd(cnt, n_in);
    if ((size_t)blockIdx.x * FIN_THREADS < (size_t)m) {
        int e = 0;
#pragma unroll
        for (int i = 0; i < 9; i++)
#pragma unroll
            for (int j = i; j < 9; j++) {
                double x = v[i] * v[j];
                for (int o = 16; o > 0; o >>= 1) x += __shfl_down_sync(0xffffffffu, x, o);
                if (lane == 0) red[wid][e] = x;
                e++;
            }
        __syncthreads();
        if (threadIdx.x < 45) {
            double x = 0.0;
            for (int w = 0; w < FIN_THREADS / 32; w++) x += red[w][threadIdx.x];
            P[(size_t)blockIdx.x * 45 + threadIdx.x] = x;
        }
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(cnt + 1, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    // five interleaved partial sums per entry (225 threads, loads batched: a single chain of ~200 dependent L2 round
    // trips cost 70 us here), combined in a fixed order: deterministic
    const int nb = (m + FIN_THREADS - 1) / FIN_THREADS;
    double* part = &red[0][0];                                    // 5 x 45 doubles, the reduction buffer is free again
    if (threadIdx.x < 225) {
        const int e = threadIdx.x % 45, g = threadIdx.x / 45;
        double x = 0.0;
#pragma unroll 8
        for (int b = g; b < nb; b += 5) x += __ldcg(&P[(size_t)b * 45 + e]);
        part[g * 45 + e] = x;
    }
    __syncthreads();
    if (threadIdx.x < 45) Gs[threadIdx.x] = (((part[threadIdx.x] + part[45 + threadIdx.x]) + part[90 + threadIdx.x]) + part[135 + threadIdx.x]) + part[180 + threadIdx.x];
    __syncthreads();
    if (threadIdx.x >= 32) return;
    if (threadIdx.x == 0) jacobi = !refit_inverse_iteration(Gs, Eb, out->E_refit, out->pose);
    __syncwarp();
    if (jacobi) solve1_warp<true>(s1, Gs, 30, out->E_refit, out->pose);      // warp-uniform
    if (threadIdx.x != 0) return;
    {
        const uint64_t packed = *packed_dev;
        out->packed = packed;
        out->hyp_id = 0xFFFFFFFFull - (packed & 0xFFFFFFFFull);
        out->count = (int32_t)(packed >> 32);
        out->n_refit = *reinterpret_cast<volatile int32_t*>(cnt);
        for (int i = 0; i < 9; i++) out->E_best[i] = Eb[i];
    }
}

// ------------------------------------------------------------------ consensus pick (eight_point.cpp:117-149)
// single block.  pose: H x 12.  Builds the candidate list in hypothesis order (R1 then R2),
// then each thread owns one candidate: distances to all, sort, trimmed mean; arg-min.
__global__ void consensus_kernel(const float* __restrict__ pose, int H, float* __restrict__ candR,
                                 float* __restrict__ candT, double* __restrict__ scratch /* C x C */,
                                 double* __restrict__ dist, int32_t* __restrict__ out /* [0]=C, [1]=chosen */)
{
    __shared__ int C_sh;
    if (threadIdx.x == 0) {
        int C = 0;
        for (int h = 0; h < H; h++) {
            const float* p = pose + (size_t)h * ERP_POSE_FLOATS;
            if (p[9] != 0.f) { for (int k = 0; k < 3; k++) { candR[3 * C + k] = p[k]; candT[3 * C + k] = p[6 + k]; } C++; }
            if (p[10] != 0.f) { for (int k = 0; k < 3; k++) { candR[3 * C + k] = p[3 + k]; candT[3 * C + k] = p[6 + k]; } C++; }
        }
        C_sh = C;
        out[0] = C;
    }
    __syncthreads();
    const int C = C_sh;
    for (int i = threadIdx.x; i < C; i += blockDim.x) {
        double* row = scratch + (size_t)i * C;
        for (int j = 0; j < C; j++) {
            float d0 = __fsub_rn(candR[3 * i], candR[3 * j]), d1 = __fsub_rn(candR[3 * i + 1], candR[3 * j + 1]);
            float d2 = __fsub_rn(candR[3 * i + 2], candR[3 * j + 2]);
            float ss = __fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2));
            row[j] = (double)__fsqrt_rn(ss);
        }
        // shell sort ascending
        for (int gap = C / 2; gap > 0; gap /= 2)
            for (int a = gap; a < C; a++) {
                double x = row[a];
                int b = a;
                for (; b >= gap && row[b - gap] > x; b -= gap) row[b] = row[b - gap];
                row[b] = x;
            }
        int lo = (int)(C * 0.2), hi = (int)(C * 0.8);
        double acc = 0.0;
        for (int j = lo; j < hi; j++) acc += row[j];
        dist[i] = acc / ((hi - lo) * 1.0);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int best = C > 0 ? 0 : -1;
        for (int i = 1; i < C; i++) if (dist[i] < dist[best]) best = i;
        out[1] = best;
    }
}

} // namespace erp

using namespace erp;

// ======================================================================================
// device-level API
// ======================================================================================
ERP_API int erp_bearings_dev(erp_ctx* ctx, const void* d_xy, size_t stride_bytes, int n,
                             int width, int height, double* d_out3, float* d_out4)
{
    ERP_ARG(ctx && n >= 0 && width > 0 && height > 0 && stride_bytes >= 8 && stride_bytes % 4 == 0, ERP_E_ARG,
            "erp_bearings_dev: bad argument");
    if (n == 0) return ERP_OK;
    ERP_ARG(d_xy && (d_out3 || d_out4), ERP_E_ARG, "erp_bearings_dev: null buffer");
    DeviceGuard g(ctx->device);
    bearings_kernel<<<cdiv(n, 256), 256, 0, ctx->stream>>>((const char*)d_xy, stride_bytes, n, width, height,
                                                          d_out3, (float4*)d_out4);
    ERP_LAUNCH(ctx, "bearings_kernel");
    return ERP_OK;
}

ERP_API int erp_gather_bearings_dev(erp_ctx* ctx, const erp_dmatch* d_matches, int n,
                                    const void* d_left_xy, const void* d_right_xy, size_t stride_bytes,
                                    int q_offset, int width, int height,
                                    double* d_l3, double* d_r3, float* d_l4, float* d_r4)
{
    ERP_ARG(ctx && n >= 0 && width > 0 && height > 0 && stride_bytes >= 8 && stride_bytes % 4 == 0, ERP_E_ARG,
            "erp_gather_bearings_dev: bad argument");
    if (n == 0) return ERP_OK;
    ERP_ARG(d_matches && d_left_xy && d_right_xy, ERP_E_ARG, "erp_gather_bearings_dev: null buffer");
    DeviceGuard g(ctx->device);
    gather_bearings_kernel<<<cdiv(n, 256), 256, 0, ctx->stream>>>(d_matches, n, nullptr, (const char*)d_left_xy, (const char*)d_right_xy,
                                                                 stride_bytes, q_offset, width, height, d_l3, d_r3,
                                                                 (float4*)d_l4, (float4*)d_r4, nullptr, nullptr);
    ERP_LAUNCH(ctx, "gather_bearings_kernel");
    return ERP_OK;
}

ERP_API int erp_pack_float4_dev(erp_ctx* ctx, const double* d_v3, int n, float* d_v4)
{
    ERP_ARG(ctx && n >= 0, ERP_E_ARG, "erp_pack_float4_dev: bad argument");
    if (n == 0) return ERP_OK;
    DeviceGuard g(ctx->device);
    pack4_kernel<<<cdiv(n, 256), 256, 0, ctx->stream>>>(d_v3, n, (float4*)d_v4);
    ERP_LAUNCH(ctx, "pack4_kernel");
    return ERP_OK;
}

namespace erp {

// gather of the matched keypoints + bearings with the match count on the device; Ks / w: also the correspondence
// operand of the tensor-core search (w must have been cleared)
int gather_bearings_chain(erp_ctx* ctx, const erp_dmatch* d_matches, int n_cap, const int32_t* d_n, const void* d_left_xy,
                          const void* d_right_xy, size_t stride, int q_offset, int W, int H, double* d_l3, double* d_r3,
                          float* d_l4, float* d_r4, float* Ks, int32_t* w)
{
    if (n_cap <= 0) return ERP_OK;
    gather_bearings_kernel<<<cdiv(n_cap, 256), 256, 0, ctx->stream>>>(d_matches, n_cap, d_n, (const char*)d_left_xy, (const char*)d_right_xy,
                                                                     stride, q_offset, W, H, d_l3, d_r3, (float4*)d_l4, (float4*)d_r4, Ks, w);
    ERP_LAUNCH(ctx, "gather_bearings_kernel");
    return ERP_OK;
}

int gather_slots_chain(erp_ctx* ctx, const erp_dmatch* d_slots, int n_ranks, int slot_records, int n_cap, erp_dmatch* d_out,
                       int32_t* d_n_out, const void* d_left_xy, const void* d_right_xy, size_t stride, int W, int H,
                       double* d_l3, double* d_r3, float* d_l4, float* d_r4, float* Ks, int32_t* w, uint32_t* ctl, const uint32_t* slot_flag)
{
    if (n_ranks > GATHER_MAX_RANKS) { set_error("more than %d ranks", GATHER_MAX_RANKS); return ERP_E_LIMIT; }
    gather_slots_kernel<<<max(1, cdiv(n_cap, 256)), 256, 0, ctx->stream>>>(d_slots, n_ranks, slot_records, n_cap, d_out, d_n_out,
                                                                          (const char*)d_left_xy, (const char*)d_right_xy, stride, W, H,
                                                                          d_l3, d_r3, (float4*)d_l4, (float4*)d_r4, Ks, w, ctl, slot_flag);
    ERP_LAUNCH(ctx, "gather_slots_kernel");
    return ERP_OK;
}

int bearings_pair_chain(erp_ctx* ctx, const void* d_left_xy, const void* d_right_xy, size_t stride, int n, int W, int H,
                        double* d_l3, double* d_r3, float* d_l4, float* d_r4, float* Ks, int32_t* w)
{
    if (n <= 0) return ERP_OK;
    bearings_pair_kernel<<<cdiv(n, 256), 256, 0, ctx->stream>>>((const char*)d_left_xy, (const char*)d_right_xy, stride, n, W, H,
                                                               d_l3, d_r3, (float4*)d_l4, (float4*)d_r4, Ks, w);
    ERP_LAUNCH(ctx, "bearings_pair_kernel");
    return ERP_OK;
}

// G for H hypotheses into d_G (H x 45)
int gram_batch(erp_ctx* ctx, const double* d_l3, const double* d_r3, int m, const int32_t* d_m, const int32_t* d_samples,
               int H, int S, uint64_t seed, uint64_t hyp0, const uint64_t* d_packed, double* d_G)
{
    if (S <= SMALL_S) {
        gram_small_kernel<<<cdiv(H, GW), GW * 32, 0, ctx->stream>>>(d_l3, d_r3, m, d_m, d_samples, H, S, seed, hyp0, d_packed, d_G);
        ERP_LAUNCH(ctx, "gram_small_kernel");
        return ERP_OK;
    }
    // large samples need an explicit table
    int slices = max(1, min(cdiv(S, GL_THREADS * 4), max(1, (ctx->sm_count * 4) / max(H, 1))));
    int st = ERP_OK;
    double* P = ctx->scratch<double>(S_PARTIAL, (size_t)H * slices * 45, &st);
    ERP_TRY(st);
    gram_large_kernel<<<dim3(slices, H), GL_THREADS, 0, ctx->stream>>>(d_l3, d_r3, m, d_samples, S, nullptr, P);
    ERP_LAUNCH(ctx, "gram_large_kernel");
    gram_finish_kernel<<<cdiv(H * 45, 256), 256, 0, ctx->stream>>>(P, H, slices, d_G);
    ERP_LAUNCH(ctx, "gram_finish_kernel");
    return ERP_OK;
}

int gram_masked(erp_ctx* ctx, const double* d_l3, const double* d_r3, int m, const uint8_t* d_mask, double* d_G)
{
    int slices = max(1, min(cdiv(m, GL_THREADS * 2), ctx->sm_count * 2));
    int st = ERP_OK;
    double* P = ctx->scratch<double>(S_PARTIAL, (size_t)slices * 45, &st);
    ERP_TRY(st);
    gram_large_kernel<<<dim3(slices, 1), GL_THREADS, 0, ctx->stream>>>(d_l3, d_r3, m, nullptr, m, d_mask, P);
    ERP_LAUNCH(ctx, "gram_large_kernel");
    gram_finish_kernel<<<1, 64, 0, ctx->stream>>>(P, 1, slices, d_G);
    ERP_LAUNCH(ctx, "gram_finish_kernel");
    return ERP_OK;
}

// max_sweeps: OpenCV's Jacobi allows 30; on a Gram matrix the relative off-diagonal test rarely fires once
// the rotations only churn rounding noise, so callers that solve ONE matrix on one thread (the RANSAC
// refit: a serial chain of ~36 rotations per sweep) cap it -- cyclic Jacobi converges quadratically and
// is at machine precision after 6-8 sweeps.
int solve_batch(erp_ctx* ctx, const double* d_G, int H, double* d_E, float* d_pose, int max_sweeps = 30)
{
    if (H == 1) {      // a single problem: one warp instead of one thread
        if (d_pose) solve1_kernel<true><<<1, 32, 0, ctx->stream>>>(d_G, max_sweeps, d_E, d_pose);
        else solve1_kernel<false><<<1, 32, 0, ctx->stream>>>(d_G, max_sweeps, d_E, nullptr);
        ERP_LAUNCH(ctx, "solve1_kernel");
        return ERP_OK;
    }
    if (d_pose) solve_kernel<true><<<cdiv(H, SOLVE_THREADS), SOLVE_THREADS, 0, ctx->stream>>>(d_G, H, max_sweeps, d_E, d_pose);
    else solve_kernel<false><<<cdiv(H, SOLVE_THREADS), SOLVE_THREADS, 0, ctx->stream>>>(d_G, H, max_sweeps, d_E, nullptr);
    ERP_LAUNCH(ctx, "solve_kernel");
    return ERP_OK;
}

// minimal samples (S = 8): sample, solve and project in one kernel
int solve_min8(erp_ctx* ctx, const double* d_l3, const double* d_r3, int m, const int32_t* d_m, const int32_t* d_samples, int H,
               uint64_t seed, uint64_t hyp0, const uint64_t* d_packed, double* d_E, float* d_pose, const Min8Fused* fused)
{
    if (H <= 0) return ERP_OK;
    Min8Fused f;
    if (fused) f = *fused;
    if (d_pose) min8_kernel<true><<<cdiv(H, MIN8_THREADS), MIN8_THREADS, 0, ctx->stream>>>(d_l3, d_r3, m, d_m, d_samples, H, seed, hyp0, d_packed, d_E, d_pose, f);
    else min8_kernel<false><<<cdiv(H, MIN8_THREADS), MIN8_THREADS, 0, ctx->stream>>>(d_l3, d_r3, m, d_m, d_samples, H, seed, hyp0, d_packed, d_E, nullptr, f);
    ERP_LAUNCH(ctx, "min8_kernel");
    return ERP_OK;
}

int finish_launch(erp_ctx* ctx, const double* d_Eb, const uint64_t* d_packed, const double* d_l3, const double* d_r3,
                  const float* d_l4, const float* d_r4, int m_cap, const int32_t* d_m, int metric, float tau, float tau2, float sin2,
                  uint8_t* d_mask, erp_ransac_result* d_result)
{
    const int grid = max(1, cdiv(m_cap, FIN_THREADS));
    int st = ERP_OK;
    double* P = ctx->scratch<double>(S_PARTIAL, (size_t)grid * 45 + 2, &st);
    ERP_TRY(st);
    int32_t* cnt = reinterpret_cast<int32_t*>(P + (size_t)grid * 45);
    ERP_CUDA(cudaMemsetAsync(cnt, 0, 2 * sizeof(int32_t), ctx->stream));
    const float4 *l4 = (const float4*)d_l4, *r4 = (const float4*)d_r4;
    switch (metric) {
    case ERP_METRIC_ALGEBRAIC: finish_kernel<ERP_METRIC_ALGEBRAIC><<<grid, FIN_THREADS, 0, ctx->stream>>>(d_Eb, d_packed, d_l3, d_r3, l4, r4, m_cap, d_m, tau, tau2, sin2, d_mask, P, cnt, d_result); break;
    case ERP_METRIC_SAMPSON: finish_kernel<ERP_METRIC_SAMPSON><<<grid, FIN_THREADS, 0, ctx->stream>>>(d_Eb, d_packed, d_l3, d_r3, l4, r4, m_cap, d_m, tau, tau2, sin2, d_mask, P, cnt, d_result); break;
    default: finish_kernel<ERP_METRIC_ANGULAR><<<grid, FIN_THREADS, 0, ctx->stream>>>(d_Eb, d_packed, d_l3, d_r3, l4, r4, m_cap, d_m, tau, tau2, sin2, d_mask, P, cnt, d_result); break;
    }
    ERP_LAUNCH(ctx, "finish_kernel");
    return ERP_OK;
}

int consensus(erp_ctx* ctx, const float* d_pose, int H, float* d_candR, float* d_candT, int32_t* d_out)
{
    int st = ERP_OK;
    size_t C = (size_t)2 * H;
    double* scr = ctx->scratch<double>(S_CONS, C * C + C, &st);
    ERP_TRY(st);
    consensus_kernel<<<1, 256, 0, ctx->stream>>>(d_pose, H, d_candR, d_candT, scr, scr + C * C, d_out);
    ERP_LAUNCH(ctx, "consensus_kernel");
    return ERP_OK;
}

} // namespace erp

ERP_API int erp_eight_point_batch_dev(erp_ctx* ctx, const double* d_l3, const double* d_r3, int m,
                                      const int32_t* d_samples, int H, int S, uint64_t seed,
                                      uint64_t hyp_offset, double* d_E, float* d_pose)
{
    ERP_ARG(ctx && d_l3 && d_r3 && d_E && H >= 0 && m >= 0, ERP_E_ARG, "erp_eight_point_batch_dev: bad argument");
    ERP_ARG(S >= 8, ERP_E_TOO_FEW_POINTS, "erp_eight_point_batch_dev: sample size %d < 8", S);
    ERP_ARG(m >= S, ERP_E_TOO_FEW_POINTS, "erp_eight_point_batch_dev: %d correspondences < sample size %d", m, S);
    ERP_ARG(d_samples || S <= SMALL_S, ERP_E_ARG, "erp_eight_point_batch_dev: samples table required for S > %d", SMALL_S);
    if (H == 0) return ERP_OK;
    DeviceGuard g(ctx->device);
    if (S == 8) return solve_min8(ctx, d_l3, d_r3, m, nullptr, d_samples, H, seed, hyp_offset, nullptr, d_E, d_pose, nullptr);
    int st = ERP_OK;
    double* G = ctx->scratch<double>(S_GRAM, (size_t)H * 45, &st);
    ERP_TRY(st);
    ERP_TRY(gram_batch(ctx, d_l3, d_r3, m, nullptr, d_samples, H, S, seed, hyp_offset, nullptr, G));
    ERP_TRY(solve_batch(ctx, G, H, d_E, d_pose));
    return ERP_OK;
}

ERP_API int erp_philox_samples(erp_ctx* ctx, uint64_t seed, uint64_t hyp_offset, int H, int S, int m, int32_t* out)
{
    ERP_ARG(ctx && out && H >= 0 && S >= 1 && S <= SMALL_S, ERP_E_ARG, "erp_philox_samples: bad argument");
    ERP_ARG(m >= S, ERP_E_TOO_FEW_POINTS, "erp_philox_samples: m %d < S %d", m, S);
    if (H == 0) return ERP_OK;
    DeviceGuard g(ctx->device);
    int st = ERP_OK;
    int32_t* d = ctx->scratch<int32_t>(S_SAMPLES, (size_t)H * S, &st);
    ERP_TRY(st);
    philox_table_kernel<<<cdiv(H, 128), 128, 0, ctx->stream>>>(seed, hyp_offset, H, S, m, d);
    ERP_LAUNCH(ctx, "philox_table_kernel");
    ERP_CUDA(cudaMemcpyAsync(out, d, sizeof(int32_t) * (size_t)H * S, cudaMemcpyDeviceToHost, ctx->stream));
    ERP_CUDA(cudaStreamSynchronize(ctx->stream));
    return ERP_OK;
}
