/*
 * erp_b200.h -- C ABI of the B200-native ERP match + eight-point hot path.
 *
 * This is the drop-in boundary.  The reference has no FFI of its own: its callers
 * include plain C++ classes (src/feature_matcher.hpp, src/eight_point.hpp,
 * src/epipolar_tool.hpp).  The class wrappers under host/ keep those signatures
 * verbatim and call the functions below; each entry point cites the reference
 * interface it replaces (paths relative to /root/reference).
 *
 * Conventions
 *  - every function returns an erp_status: 0 ok, > 0 argument/domain error,
 *    < 0 CUDA failure.  erp_last_error() gives the message (thread local).
 *  - there is NO CPU fallback: without a CUDA device erp_ctx_create fails.
 *  - "host" entry points take borrowed host pointers and copy through
 *    context-owned staging buffers; "_dev" entry points take device pointers,
 *    enqueue on the context stream and do not synchronise unless stated.
 *  - row-major, little endian.  fp32 descriptors, fp64 bearings (cv::Point3d),
 *    erp_dmatch has the layout of cv::DMatch (16 bytes).
 *  - one context per host thread and device; a context is not thread safe.
 */
#ifndef ERP_B200_H
#define ERP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ERP_B200_VERSION 200

typedef struct erp_ctx erp_ctx;

typedef struct {          /* == cv::DMatch */
    int32_t queryIdx;
    int32_t trainIdx;
    int32_t imgIdx;
    float distance;
} erp_dmatch;

typedef enum {
    ERP_OK = 0,
    ERP_E_ARG = 1,             /* null pointer, negative size, bad stride ...                  */
    ERP_E_DIM = 2,             /* descriptor dimension not a positive multiple of 4, > 512      */
    ERP_E_TOO_FEW_TRAIN = 3,   /* k=2 needs >= 2 train rows (the reference throws / is UB)      */
    ERP_E_TOO_FEW_POINTS = 4,  /* fewer correspondences than the sample size                    */
    ERP_E_NO_CANDIDATE = 5,    /* initial_guess: no hypothesis passed the <1.57 rad test (UB in ref) */
    ERP_E_LIMIT = 6,           /* a size exceeds an implementation limit                        */
    ERP_E_CUDA = -1,
    ERP_E_NO_DEVICE = -2,
    ERP_E_ARCH = -3,           /* device is not sm_100                                          */
    ERP_E_NCCL = -4            /* NCCL missing (libnccl.so.2 not loadable) or a collective failed */
} erp_status;

typedef enum {
    ERP_METRIC_ALGEBRAIC = 0,  /* |l^T E r| < tau          (src/epipolar_tool.cpp:100-107, tau 0.002) */
    ERP_METRIC_SAMPSON = 1,    /* res^2 < tau^2 (|E r|^2 + |E^T l|^2)                             */
    ERP_METRIC_ANGULAR = 2     /* angle(l, epipolar plane of r) < tau   (one_image_test/main.cpp:27-50) */
} erp_metric;

/* which distance engine erp_knn2* uses */
typedef enum {
    ERP_ENGINE_AUTO = 0,       /* the fastest exact engine for the shape: TCGEN05_1X for large problems, else SIMT */
    ERP_ENGINE_EXACT_SIMT = 1, /* fp64 direct-form brute force (also the rescan path)            */
    ERP_ENGINE_TCGEN05 = 2,    /* 3xTF32 GEMM-form tiles + fused top-4, exact fp64 refine + certificate  */
    ERP_ENGINE_TCGEN05_1X = 3  /* one product of f16 operands (11 significant bits), top-8, same certificate:
                                  5 tensor instructions per tile at D = 64 where 3xTF32 issues 24 */
} erp_engine;

/* operand format of the tensor products of a distance search (erp_ctx_last_knn_operands) */
typedef enum {
    ERP_OPERANDS_NONE = 0,     /* no tensor product: ERP_ENGINE_EXACT_SIMT */
    ERP_OPERANDS_TF32 = 1,
    ERP_OPERANDS_F16 = 2,
    ERP_OPERANDS_I8 = 3        /* binary descriptors: bits expanded to +-1 int8, tcgen05.mma.kind::i8, exact s32 */
} erp_operands;

/* pose record per hypothesis: XYZ-euler of R1, of R2 (rad), t, validity flags (1.0/0.0), 1 pad */
#define ERP_POSE_FLOATS 12

typedef struct {
    uint64_t packed;        /* (count << 32) | (0xFFFFFFFF - hyp_id): max == best, ties -> lowest id */
    uint64_t hyp_id;
    int32_t  count;         /* inliers of the winning hypothesis (fp32 scoring)                */
    int32_t  n_refit;       /* correspondences used by the refit (== count)                    */
    double   E_best[9];     /* rank-2 corrected E of the winning minimal sample                */
    double   E_refit[9];    /* least-squares eight-point on its inliers (eight_point.cpp:16-50) */
    float    pose[ERP_POSE_FLOATS]; /* decomposition of E_refit                                */
} erp_ransac_result;

/* ---------------------------------------------------------------- context */
const char* erp_last_error(void);
int  erp_version(void);
int  erp_device_count(void);
int  erp_ctx_create(int device, erp_ctx** out);
void erp_ctx_destroy(erp_ctx* ctx);
void* erp_ctx_stream(erp_ctx* ctx);                 /* cudaStream_t the context enqueues on */
int  erp_ctx_synchronize(erp_ctx* ctx);
int  erp_ctx_set_engine(erp_ctx* ctx, int engine);  /* erp_engine */
int  erp_ctx_device(erp_ctx* ctx);
/* number of kernels this context has launched since creation (bench "gpu_launches") */
uint64_t erp_ctx_launch_count(erp_ctx* ctx);
/* diagnostics of the last erp_knn2* call: [0] engine used, [1] queries re-scanned exactly, and the plan of the distance
 * kernel: [2] segments per query row (each writes its own candidate lists), [3] units (query tile x train tile) per CTA,
 * [4] CTAs.  The SIMT engines report 1, their query blocks and 0.  After a tensor-core search of float rows, [4] is
 * instead the largest observed |approximate - exact| / (|q|^2 + max|t|^2) of a candidate score, in 1e-12 units. */
int  erp_ctx_last_knn_stats(erp_ctx* ctx, int64_t out[5]);
/* operands of the last erp_knn2* call: [0] erp_operands, and for f16 operands [1] 1 if the range guard fired (a finite input
 * f16 cannot hold: every query of the call was re-scanned exactly), [2] queries re-scanned because f16 could not represent
 * them closely enough (the guard, or norms so small that subnormal rounding is outside the certificate); synchronises */
int  erp_ctx_last_knn_operands(erp_ctx* ctx, int64_t out[3]);
/* device time of the dominant distance kernel of the last erp_knn2* call, from CUDA events the
 * library records on its own stream around that launch (synchronises the stream) */
int  erp_ctx_last_knn_kernel_ms(erp_ctx* ctx, float* ms);
/* summed device time of the hypothesis-scoring kernel launches of the last erp_ransac_local_dev /
 * erp_ransac call (same event mechanism); *launches (optional) = how many launches that was */
int  erp_ctx_last_score_kernel_ms(erp_ctx* ctx, float* ms, int* launches);
/* the last tensor-core best-hypothesis search (last chunk of the last RANSAC call): [0] hypotheses,
 * [1] correspondence tiles (256 each) every hypothesis was bounded on, [2] tiles in total,
 * [3] survivors bounded on the remaining tiles, [4] contenders scored exactly, [5] L* */
int  erp_ctx_last_score_stats(erp_ctx* ctx, int64_t out[6]);
/* device time of the stages of the last erp_pair_pose* call on this context, from CUDA events on its stream:
 * [0] matching (2-NN, certificate, ratio / cross-check filter), [1] match exchange (multi-GPU all-gather) + gather of
 * the matched keypoints + bearings, [2] RANSAC (sample, solve, score, best-model reduction, mask, refit) */
int  erp_ctx_last_stage_ms(erp_ctx* ctx, float out[3]);

/* ---------------------------------------------------------------- matching
 * replaces feature_matcher::match_two_image      src/feature_matcher.hpp:36, .cpp:42-59
 *          cv::DescriptorMatcher::knnMatch(k=2)  src/feature_matcher.cpp:45
 * ratio < 0 disables the ratio test; the reference uses 0.3f (.cpp:47).
 * cross_check != 0 additionally keeps (q,t) only if q is t's nearest query
 * (cv::BFMatcher(crossCheck=true) semantics; an extension, SURVEY D5).
 * Strides are in bytes between rows (cv::Mat::step).  out needs room for nq records. */
int erp_knn2_match(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes,
                   const float* t, int nt, size_t t_stride_bytes, int dim,
                   float ratio, int cross_check, erp_dmatch* out, int* n_out);
/* raw 2-NN: idx2 / dist2 are nq x 2 (nearest first); either may be NULL */
int erp_knn2_raw(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes,
                 const float* t, int nt, size_t t_stride_bytes, int dim,
                 int32_t* idx2, float* dist2);

/* Near-tie report (diagnostic; north_star: "bit-exact except for documented fp32 distance ties within 1e-6 relative").
 * The 2-NN above is exact (fp64 distances); the reference compares fp32 distances (src/feature_matcher.cpp:45,52), so
 * an fp32 matcher may legitimately return another index where two distances are closer than its rounding error.
 * flags[i] for query i: bit 0 = the two nearest are within rel_tol of each other (|d1 - d0| <= rel_tol * d1: their
 * ORDER may differ), bit 1 = a third train row is within rel_tol of the second (d <= d1 (1 + rel_tol): the second
 * INDEX may differ).  Exact fp64 brute force over all pairs; flags: nq bytes, *n_flagged = how many are non-zero. */
int erp_knn2_near_ties(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes,
                       const float* t, int nt, size_t t_stride_bytes, int dim, float rel_tol,
                       uint8_t* flags, int* n_flagged);

/* device-resident forms (dense rows: stride == dim * 4) */
int erp_knn2_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                 int32_t* d_idx2, float* d_dist2, double* d_d2 /* nq x 2 or NULL */);
/* nearest query per train row over this rank's queries; indices offset by q_offset.
 * d_best_d2 (nt doubles) and d_best_q (nt int32) feed the multi-GPU min-reduction. */
int erp_nn1_reverse_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                        int q_offset, int32_t* d_best_q, double* d_best_d2);
/* ratio + (optional) cross-check filter with ordered compaction (feature_matcher.cpp:50-56).
 * d_rev_best_q: nt global query ids or NULL.  d_n_out: one int32 on the device. */
int erp_match_filter_dev(erp_ctx* ctx, const int32_t* d_idx2, const float* d_dist2, int nq,
                         float ratio, const int32_t* d_rev_best_q, int q_offset,
                         erp_dmatch* d_out, int32_t* d_n_out);
/* the three above chained on one device */
int erp_knn2_match_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim,
                       float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out);

/* ---------------------------------------------------------------- binary descriptors
 * replaces feature_matcher::match_two_image      src/feature_matcher.cpp:42-59
 * with cv::BFMatcher(NORM_HAMMING) in place of the L2 matcher: ORB, AKAZE (MLDB), BRISK, FREAK, LATCH rows.
 * Rows are nbytes uint8 (1 <= nbytes <= 64, else ERP_E_DIM), strides in bytes; distance = popcount(q XOR t) over the
 * nbytes bytes, carried as a float in erp_dmatch.distance and dist2 (as NORM_HAMMING does).  2-NN order is (distance,
 * trainIdx) ascending: exact ties go to the lowest trainIdx.  Ratio test, cross-check (reverse ties: lowest queryIdx)
 * and output order are those of the float entry points.  Every engine returns the same bits:
 *   ERP_ENGINE_EXACT_SIMT              __popc on 32-bit words
 *   ERP_ENGINE_TCGEN05, _TCGEN05_1X    both select the tcgen05.mma.kind::i8 engine (bits as +-1 int8: dot = n - 2 H,
 *                                      exact in the s32 accumulator, so there is nothing to certify or re-scan)
 *   ERP_ENGINE_AUTO                    kind::i8 from 1e6 query x train pairs up, SIMT below
 * erp_ctx_last_knn_stats: [0] engine, [1] 0 (never re-scanned); erp_ctx_last_knn_operands: ERP_OPERANDS_I8 or NONE.
 * Not provided for binary rows: the multi-GPU forms (_dist, erp_group_*). */
int erp_knn2_match_bin(erp_ctx* ctx, const uint8_t* q, int nq, size_t q_stride_bytes,
                       const uint8_t* t, int nt, size_t t_stride_bytes, int nbytes,
                       float ratio, int cross_check, erp_dmatch* out, int* n_out);
int erp_knn2_raw_bin(erp_ctx* ctx, const uint8_t* q, int nq, size_t q_stride_bytes,
                     const uint8_t* t, int nt, size_t t_stride_bytes, int nbytes,
                     int32_t* idx2, float* dist2);
/* device-resident forms (dense rows: stride == nbytes), enqueue only */
int erp_knn2_bin_dev(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes,
                     int32_t* d_idx2, float* d_dist2, double* d_d2 /* nq x 2 or NULL */);
int erp_knn2_match_bin_dev(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes,
                           float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out);

/* ---------------------------------------------------------------- geometry
 * pixel -> unit-sphere bearing, replaces src/eight_point.cpp:157-186.
 * xy points at the first (x,y) float pair; stride 28 == sizeof(cv::KeyPoint). */
int erp_bearings_from_pixels(erp_ctx* ctx, const void* xy, size_t stride_bytes, int n,
                             int width, int height, double* out3);
int erp_bearings_dev(erp_ctx* ctx, const void* d_xy, size_t stride_bytes, int n,
                     int width, int height, double* d_out3, float* d_out4 /* n x 4 or NULL */);
/* gather + convert: for match i, left bearing of keypoint queryIdx and right bearing of keypoint
 * trainIdx (src/spherical_surf.cpp:155-162 followed by src/eight_point.cpp:163-186), fused.
 * q_offset is subtracted from queryIdx when left_xy holds only this rank's shard. */
int erp_gather_bearings_dev(erp_ctx* ctx, const erp_dmatch* d_matches, int n,
                            const void* d_left_xy, const void* d_right_xy, size_t stride_bytes,
                            int q_offset, int width, int height,
                            double* d_l3, double* d_r3, float* d_l4, float* d_r4);
/* fp64 n x 3 -> fp32 n x 4 copies used by scoring */
int erp_pack_float4_dev(erp_ctx* ctx, const double* d_v3, int n, float* d_v4);

/* batched hypothesis solve, replaces eight_point::eight_point_estimation per hypothesis
 * (src/eight_point.cpp:16-85).  samples: H x S indices into the m correspondences, or NULL
 * to draw S distinct indices per hypothesis with Philox4x32-10 keyed by (seed, hyp_offset+h).
 * E_out: H x 9 rank-2 corrected E (l^T E r = 0, row major).  pose_out: H x 12 or NULL. */
int erp_eight_point_batch(erp_ctx* ctx, const double* l3, const double* r3, int m,
                          const int32_t* samples, int H, int S, uint64_t seed, uint64_t hyp_offset,
                          double* E_out, float* pose_out);
int erp_eight_point_batch_dev(erp_ctx* ctx, const double* d_l3, const double* d_r3, int m,
                              const int32_t* d_samples, int H, int S, uint64_t seed,
                              uint64_t hyp_offset, double* d_E, float* d_pose);
/* the Philox sample table alone (for replay by the oracle): out H x S */
int erp_philox_samples(erp_ctx* ctx, uint64_t seed, uint64_t hyp_offset, int H, int S, int m,
                       int32_t* out);

/* eight_point::eight_point_estimation called directly on n >= 8 correspondences
 * (src/manual.cpp:152): the N-point least-squares solve, also used as the refit. */
int erp_eight_point_estimation(erp_ctx* ctx, const double* l3, const double* r3, int n,
                               double* E_out /* 9 or NULL */, float* R1_vec, float* R2_vec,
                               float* T_vec, int* R1_valid, int* R2_valid);

/* ---------------------------------------------------------------- scoring / RANSAC
 * residual of src/epipolar_tool.cpp:100-107 over all correspondences per hypothesis */
int erp_score(erp_ctx* ctx, const double* E, int H, const double* l3, const double* r3, int m,
              int metric, float tau, int32_t* counts);
int erp_score_dev(erp_ctx* ctx, const double* d_E, int H, const float* d_l4, const float* d_r4,
                  int m, int metric, float tau, uint64_t hyp_offset,
                  int32_t* d_counts /* H or NULL */, uint64_t* d_best_packed /* 1, max-merged, or NULL */);
int erp_inlier_mask(erp_ctx* ctx, const double* E9, const double* l3, const double* r3, int m,
                    int metric, float tau, uint8_t* mask, int* n_inliers);
/* least-squares refit on mask != 0 (mask NULL = all points) */
int erp_refit(erp_ctx* ctx, const double* l3, const double* r3, int m, const uint8_t* mask,
              double* E_out, float* pose_out);

/* whole minimal-sample RANSAC on one device: hypotheses [hyp_offset, hyp_offset+H) */
int erp_ransac(erp_ctx* ctx, const double* l3, const double* r3, int m, uint64_t seed,
               uint64_t hyp_offset, int H, int S, int metric, float tau,
               erp_ransac_result* result, uint8_t* mask /* m or NULL */);
/* the same on the matched KEYPOINTS (the argument list of eight_point::find, src/eight_point.cpp:152-192, with the
 * RANSAC parameters instead of the 80-round schedule): pixels -> bearings (src/eight_point.cpp:163-186) -> RANSAC on the
 * device; the bearings never travel.  left_xy / right_xy: first two floats of every stride_bytes record (8 = packed
 * xy pairs, 28 = cv::KeyPoint). */
int erp_ransac_pixels(erp_ctx* ctx, int width, int height, const void* left_xy, const void* right_xy,
                      size_t stride_bytes, int m, uint64_t seed, uint64_t hyp_offset, int H, int S, int metric,
                      float tau, erp_ransac_result* result, uint8_t* mask /* m or NULL */);
/* One call per ERP pair -- the sequence of src/automatic.cpp:117-126 (match_two_image, gather of the matched keypoints,
 * eight_point::find) with the RANSAC schedule: descriptors and ALL keypoints of both views go up once, matches, their
 * gather, the bearings and the hypotheses stay on the device, the match records, the pose and the inlier mask come back.
 * left_xy has nq records, right_xy nt records (first two floats of every kp_stride_bytes bytes).  With fewer matches than
 * S the matches are still returned and the status is ERP_E_TOO_FEW_POINTS. */
int erp_pair_pose(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                  int dim, float ratio, int cross_check,
                  const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                  uint64_t seed, int H, int S, int metric, float tau,
                  erp_dmatch* matches_out /* nq */, int* n_matches, erp_ransac_result* result, uint8_t* mask /* nq or NULL */);
/* the same with everything on the device (dense rows, kp_stride_bytes between keypoint records) and NOTHING awaited: the
 * call only enqueues.  d_matches needs room for nq records, d_n_matches is one int32, d_mask nq bytes or NULL, d_result one
 * erp_ransac_result -- all device memory.  The match count never visits the host: every launch of the pose chain is sized
 * for nq and reads the count from d_n_matches.  With fewer than S matches the result is meaningless (check *d_n_matches). */
int erp_pair_pose_dev(erp_ctx* ctx, const float* d_q, int nq, const float* d_t, int nt, int dim, float ratio, int cross_check,
                      const void* d_left_xy, const void* d_right_xy, size_t kp_stride_bytes, int width, int height,
                      uint64_t seed, int H, int S, int metric, float tau,
                      erp_dmatch* d_matches, int32_t* d_n_matches, uint8_t* d_mask, erp_ransac_result* d_result);
/* erp_pair_pose / erp_pair_pose_dev on binary descriptors (nbytes per row, Hamming matching as erp_knn2_match_bin);
 * same keypoint, RANSAC and output arguments */
int erp_pair_pose_bin(erp_ctx* ctx, const uint8_t* q, int nq, size_t q_stride_bytes, const uint8_t* t, int nt,
                      size_t t_stride_bytes, int nbytes, float ratio, int cross_check,
                      const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                      uint64_t seed, int H, int S, int metric, float tau,
                      erp_dmatch* matches_out /* nq */, int* n_matches, erp_ransac_result* result, uint8_t* mask /* nq or NULL */);
int erp_pair_pose_bin_dev(erp_ctx* ctx, const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int nbytes, float ratio,
                          int cross_check, const void* d_left_xy, const void* d_right_xy, size_t kp_stride_bytes, int width,
                          int height, uint64_t seed, int H, int S, int metric, float tau,
                          erp_dmatch* d_matches, int32_t* d_n_matches, uint8_t* d_mask, erp_ransac_result* d_result);
/* sharded form: every rank scores its hypothesis range and leaves its packed best in
 * d_packed (one uint64 on the device); the caller max-reduces it across ranks (one 8-byte
 * NCCL allreduce) and calls erp_ransac_finish_dev with the winning packed value. */
int erp_ransac_local_dev(erp_ctx* ctx, const double* d_l3, const double* d_r3,
                         const float* d_l4, const float* d_r4, int m, uint64_t seed,
                         uint64_t hyp_offset, int H, int S, int metric, float tau,
                         uint64_t* d_packed);
int erp_ransac_finish_dev(erp_ctx* ctx, const double* d_l3, const double* d_r3,
                          const float* d_l4, const float* d_r4, int m, uint64_t seed,
                          uint64_t packed, int S, int metric, float tau,
                          uint8_t* d_mask /* m or NULL */, erp_ransac_result* result /* host */);

/* ---------------------------------------------------------------- multi-GPU (SURVEY 8e; north_star's split of ONE pair)
 * The reference is single-process CPU code (src/automatic.cpp:117-126 calls match_two_image then find): there is no
 * reference interface to cite for the split itself.  The work is cut where it is independent:
 *   - query rows  [lo, hi) = erp_shard_range(nq, rank, nranks) per GPU, train set replicated (host-buffer calls upload
 *     1/nranks of it per GPU and all-gather it over NVLink);
 *   - hypothesis ids erp_shard_range(H, rank, nranks) per GPU (Philox is keyed by the global id: results do not depend
 *     on nranks);
 * and the exchange steps are: one all-gather of the per-rank match lists (fixed-size slots, rank order = ascending
 * queryIdx), ONE 8-byte max all-reduce of the packed best model, and for cross-check a min all-reduce over the
 * per-train (d2, queryIdx).  NCCL is loaded at run time (dlopen of libnccl.so.2; the library does not link it).
 * Two ways to form the clique:
 *   a) one process per GPU (torchrun, MPI ...): rank 0 calls erp_comm_unique_id, the caller broadcasts the 128 bytes,
 *      every rank calls erp_comm_init on its own context;
 *   b) one process, several GPUs: erp_group_create(devices) builds the contexts, the clique (ncclCommInitAll) and one
 *      worker thread per device; erp_group_* calls fan out inside the call (what the C++ classes do when
 *      $ERP_B200_DEVICES names more than one device). */
#define ERP_COMM_ID_BYTES 128
int erp_shard_range(int n, int rank, int nranks, int* lo, int* hi);   /* contiguous, sizes differ by at most one */
int erp_comm_unique_id(void* id_out /* ERP_COMM_ID_BYTES */);
int erp_comm_init(erp_ctx* ctx, int nranks, int rank, const void* id /* ERP_COMM_ID_BYTES */);
int erp_comm_destroy(erp_ctx* ctx);
int erp_comm_size(erp_ctx* ctx);                                    /* 1 without a clique */
int erp_comm_rank(erp_ctx* ctx);
/* in-place max all-reduce of one packed best-model word (the single small collective of north_star) */
int erp_comm_allreduce_best_dev(erp_ctx* ctx, uint64_t* d_packed);
/* cross-check: global nearest query per train row from the per-rank results of erp_nn1_reverse_dev (min d2, then the
 * lowest query id among the ranks that attain it: cv::BFMatcher(crossCheck) tie order); in place, nt entries */
int erp_comm_cross_check_dev(erp_ctx* ctx, int32_t* d_best_q, double* d_best_d2, int nt);
/* one ERP pair split over the clique of ctx; collective: every rank calls it with the same arguments.
 * d_q_shard: this rank's query rows [lo, hi) of nq_total; d_t: all nt train rows; keypoints of ALL queries / train rows.
 * Outputs as erp_pair_pose_dev, identical on every rank (d_matches holds the concatenated list, nq_total records).
 * Only enqueues.  Without a clique it is erp_pair_pose_dev. */
int erp_pair_pose_dist_dev(erp_ctx* ctx, const float* d_q_shard, int nq_total, const float* d_t, int nt, int dim,
                           float ratio, int cross_check,
                           const void* d_left_xy, const void* d_right_xy, size_t kp_stride_bytes, int width, int height,
                           uint64_t seed, int H_total, int S, int metric, float tau,
                           erp_dmatch* d_matches, int32_t* d_n_matches, uint8_t* d_mask, erp_ransac_result* d_result);
/* host buffers, same arguments as erp_pair_pose on every rank (all ranks see the same host data): a rank uploads its
 * query shard, 1/nranks of the train rows (all-gathered on the device) and the keypoints; results on every rank. */
int erp_pair_pose_dist(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                       int dim, float ratio, int cross_check,
                       const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                       uint64_t seed, int H, int S, int metric, float tau,
                       erp_dmatch* matches_out /* nq */, int* n_matches, erp_ransac_result* result, uint8_t* mask /* nq or NULL */);
/* query-sharded feature_matcher::match_two_image (src/feature_matcher.cpp:42-59): this rank's part of the match list
 * (global query ids, ascending); the caller concatenates the parts in rank order.  out needs room for hi - lo records. */
int erp_knn2_match_dist(erp_ctx* ctx, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                        int dim, float ratio, int cross_check, erp_dmatch* out, int* n_out);

/* the same on device-resident descriptors (d_q_shard: this rank's rows of the nq_total queries), enqueue only;
 * d_out needs room for the shard's rows, d_n_out is one int32 on the device */
int erp_knn2_match_dist_dev(erp_ctx* ctx, const float* d_q_shard, int nq_total, const float* d_t, int nt, int dim,
                            float ratio, int cross_check, erp_dmatch* d_out, int32_t* d_n_out);

typedef struct erp_group erp_group;
int  erp_group_create(const int* devices, int ndev, erp_group** out);   /* ndev == 1 works without NCCL */
void erp_group_destroy(erp_group* g);
int  erp_group_size(erp_group* g);
erp_ctx* erp_group_ctx(erp_group* g, int rank);
/* erp_pair_pose / erp_knn2_match fanned out over the group's devices inside the call; same arguments and results */
int erp_group_pair_pose(erp_group* g, const float* q, int nq, size_t q_stride_bytes, const float* t, int nt, size_t t_stride_bytes,
                        int dim, float ratio, int cross_check,
                        const void* left_xy, const void* right_xy, size_t kp_stride_bytes, int width, int height,
                        uint64_t seed, int H, int S, int metric, float tau,
                        erp_dmatch* matches_out, int* n_matches, erp_ransac_result* result, uint8_t* mask);
int erp_group_knn2_match(erp_group* g, const float* q, int nq, size_t q_stride_bytes,
                         const float* t, int nt, size_t t_stride_bytes, int dim,
                         float ratio, int cross_check, erp_dmatch* out, int* n_out);

/* ---------------------------------------------------------------- rows next to the hot path (SURVEY 8f)
 * 8-bit, 3-channel images (cv::Mat CV_8UC3), strides in bytes.  Unmapped output pixels are written 0
 * (the reference leaves them uninitialised).
 * erp_rotation::rotate_image          src/erp_rotation.cpp:94-122 (inverse mapping with rot_mat.inv()) */
int erp_rotate_image(erp_ctx* ctx, const uint8_t* im, int width, int height, size_t stride_bytes,
                     const double* R9, uint8_t* out, size_t out_stride_bytes);
int erp_rotate_image_dev(erp_ctx* ctx, const uint8_t* d_im, int width, int height, size_t stride_bytes,
                         const double* R9 /* host */, uint8_t* d_out, size_t out_stride_bytes);
/* spherical_surf::crop_rotated_image  src/spherical_surf.cpp:16-48: out is (height/4) x width */
int erp_crop_rotated_image(erp_ctx* ctx, const uint8_t* im, int width, int height, size_t stride_bytes,
                           float pitch_rot_deg, uint8_t* out, size_t out_stride_bytes);
int erp_crop_rotated_image_dev(erp_ctx* ctx, const uint8_t* d_im, int width, int height, size_t stride_bytes,
                               float pitch_rot_deg, uint8_t* d_out, size_t out_stride_bytes);
/* erp_rotation::rotate_pixel          src/erp_rotation.cpp:66-92 on n (row, col) int32 pairs */
int erp_rotate_pixels(erp_ctx* ctx, const int32_t* rc, int n, const double* R9, int width, int height, int32_t* out);
/* spherical_surf::rotate_keypoint     src/spherical_surf.cpp:50-63, in place on (x, y) float pairs
 * (stride 28 == sizeof(cv::KeyPoint)) */
int erp_rotate_keypoints(erp_ctx* ctx, void* xy, size_t stride_bytes, int n, float pitch_rot_inv_deg, int width, int height);
int erp_rotate_keypoints_dev(erp_ctx* ctx, void* d_xy, size_t stride_bytes, int n, float pitch_rot_inv_deg, int width, int height);

/* epipolar_tool::draw_epipole           src/epipolar_tool.cpp:84-128 (ctor geometry :35-81 included).
 * left_xy / right_xy: HOST (x, y) float pairs of the n_key <= 7 selected correspondences (stride 28 ==
 * sizeof(cv::KeyPoint)); E9 in the tool's convention (result = l . (E^T p), |result| < 0.002).
 * Sequential loop semantics, dots clipped to the image (the reference races and writes out of bounds). */
int erp_draw_epipole(erp_ctx* ctx, const double* E9, const void* left_xy, const void* right_xy, size_t stride_bytes,
                     int n_key, int im_width, int im_height, int out_width, int out_height,
                     uint8_t* out, size_t out_stride_bytes);
int erp_draw_epipole_dev(erp_ctx* ctx, const double* E9, const void* left_xy, const void* right_xy, size_t stride_bytes,
                         int n_key, int im_width, int im_height, int out_width, int out_height,
                         uint8_t* d_out, size_t out_stride_bytes);

/* ---------------------------------------------------------------- reference mode
 * eight_point::initial_guess  src/eight_point.hpp:20-23, .cpp:87-150
 * samples: H x S table (H = 80, S = int(m*0.25) in the reference) or NULL to replay
 * libstdc++ random_shuffle over never-seeded glibc rand() (src/eight_point.hpp:54-58).
 * cand_R / cand_T: room for 2H x 3 floats, or NULL. */
int erp_initial_guess(erp_ctx* ctx, const double* l3, const double* r3, int m,
                      const int32_t* samples, int H, int S,
                      float* R_vec_out, float* T_vec_out,
                      float* cand_R, float* cand_T, int* n_cand, int* chosen);
/* eight_point::find  src/eight_point.hpp:11-14, .cpp:152-192 */
int erp_find(erp_ctx* ctx, int width, int height, const void* left_xy, const void* right_xy,
             size_t stride_bytes, int match_size, const int32_t* samples, int H, int S,
             float* R_vec_out, float* T_vec_out);
/* host-side replay of random_array (glibc TYPE_3 rand + libstdc++ shuffle): H x S */
int erp_libstdcxx_sample_table(int m, int H, int S, unsigned seed, int32_t* table);

#ifdef __cplusplus
}
#endif
#endif /* ERP_B200_H */
