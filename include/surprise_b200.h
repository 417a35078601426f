/*
 * surprise_b200 -- C-ABI of the B200-native fit-time hot path of Surprise (nickmvincent/Surprise).
 *
 * The reference has no FFI of its own: its "operator API" for this path is (i) the module-level
 * callables of surprise/similarities.pyx looked up by name in
 * surprise/prediction_algorithms/algo_base.py:269-272 and (ii) the sgd()/estimate() methods of the
 * AlgoBase subclasses in surprise/prediction_algorithms/matrix_factorization.pyx.  Every entry point
 * below replaces one of those Cython functions and says which (file:line, relative to the reference
 * root).  INTEGRATION.md shows the ctypes stub a maintainer would add on the reference side.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  No torch / numpy types.
 *   - Every function comes in two forms:
 *       sb2_<name>_dev(...,  void* stream)  all array arguments are DEVICE pointers; work is enqueued
 *                                           on `stream` (a cudaStream_t; NULL = default stream) and the
 *                                           call returns after the stream has been synchronised only
 *                                           where a status must be read back (documented per call).
 *       sb2_<name>(...)                     all array arguments are HOST pointers; the library does
 *                                           the H2D / D2H copies itself (this is the e2e boundary).
 *   - Return value: SB2_OK or an error code; sb2_last_error() gives the message of the calling
 *     thread's last failure.  There is NO CPU fallback: without a usable CUDA device every compute
 *     entry point fails with SB2_ERR_CUDA.
 *   - Index types: int32 ids, int64 CSR offsets, fp64 ratings / factors at the boundary (the reference
 *     hands Python floats / float64 ndarrays).
 *   - "yr CSR": y_ptr[n_y+1], x_idx[nnz], r[nnz] -- the flattening of the reference's
 *     `yr` dict-of-lists in iteration order (for y in yr: for (x, r) in yr[y]).
 *   - "all_ratings COO": u[n], i[n], r[n] in trainset.all_ratings() order (trainset.py:180-190).
 */
#ifndef SURPRISE_B200_H
#define SURPRISE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    SB2_OK = 0,
    SB2_ERR_CUDA = 1,          /* CUDA runtime / driver failure (includes "no device") */
    SB2_ERR_INVALID = 2,       /* bad argument */
    SB2_ERR_ZERO_DIVISION = 3, /* the reference would raise ZeroDivisionError (cdivision=False) */
    SB2_ERR_DUPLICATE = 4,     /* duplicate (x, y) pair in yr: not representable in the dense panels */
    SB2_ERR_UNSUPPORTED = 5    /* ratings not representable on the exact integer-digit path */
};

enum { SB2_SIM_COSINE = 0, SB2_SIM_MSD = 1, SB2_SIM_PEARSON = 2, SB2_SIM_PEARSON_BASELINE = 3 };

/* library / device introspection */
const char* sb2_last_error(void);
int sb2_version(void);
int sb2_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* total_mem_bytes);
/* kernels launched by this library on the calling thread since the last reset (bench: gpu_launches) */
int64_t sb2_launch_count(void);
void sb2_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Similarity matrices.  Replaces similarities.pyx:28-97 (cosine), :100-166 (msd), :169-258
 * (pearson), :261-361 (pearson_baseline), as dispatched by algo_base.py:256-301.
 *
 * Ratings must be exact multiples of 1/rating_denom with r*rating_denom an integer in [0, 65535]
 * (MovieLens stars: denom 1, half-stars: 2, Jester two-decimals: 100); they are split into base-256
 * digits and contracted on the int8 tensor cores with exact int32 accumulation.  For cosine / msd /
 * pearson the result is bit-identical to the reference whenever all the reference's partial sums
 * are exactly representable (true for every integer / half-integer scale); pearson_baseline is
 * floating point in the reference too and matches it to ~1e-12 absolute (contract: 1e-9).
 *
 * Rows [row_begin, row_end) of the n_x x n_x matrix are produced into sim_out (row-major,
 * (row_end-row_begin) x n_x): the row-block shard of one rank (row_begin a multiple of 256, the tile of the
 * CTA-pair MMA kernel).  row_begin = 0, row_end = n_x builds
 * the whole matrix and exploits symmetry.  x_biases / y_biases / global_mean / shrinkage are only
 * read for SB2_SIM_PEARSON_BASELINE (min_support is clamped to >= 2 there, similarities.pyx:334).
 * The _dev form synchronises `stream` once to read the duplicate / zero-division status.
 * ------------------------------------------------------------------------------------------------ */
int sb2_sim_build_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx,
                      const double* r, int64_t nnz, int rating_denom, int min_support, double global_mean,
                      const double* x_biases, const double* y_biases, double shrinkage, int64_t row_begin,
                      int64_t row_end, double* sim_out, void* stream);
int sb2_sim_build(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx,
                  const double* r, int64_t nnz, int rating_denom, int min_support, double global_mean,
                  const double* x_biases, const double* y_biases, double shrinkage, int64_t row_begin,
                  int64_t row_end, double* sim_out);

/* Test hook: C[m x n] (int32, row-major, ld = n) = A[m x k] * B[n x k]^T for u8 operands through the
 * tcgen05 kernel (use_tensor_cores = 1) or through the scalar dp4a cross-check kernel (0).
 * m, n multiples of 256, k multiple of 128.  Device pointers. */
int sb2_gemm_u8_selftest_dev(int use_tensor_cores, int64_t m, int64_t n, int64_t k, const uint8_t* a,
                             const uint8_t* b, int32_t* c, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Baselines.  Replaces prediction_algorithms/optimize_baselines.pyx:14-54 (baseline_als) and
 * :57-84 (baseline_sgd).  ALS is bit-exact (order-preserving segmented sums); SGD is a sequential
 * recursion and is executed as such (one thread), bit-exact but slow -- non-default in the reference.
 * ur CSR: u_ptr[n_users+1], ui_idx[n], u_r[n] (ur[u] list order); ir CSR likewise (ir[i] list order).
 * ------------------------------------------------------------------------------------------------ */
int sb2_baseline_als_dev(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx,
                         const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                         double global_mean, int n_epochs, double reg_u, double reg_i, double* bu, double* bi,
                         void* stream);
int sb2_baseline_als(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx,
                     const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                     double global_mean, int n_epochs, double reg_u, double reg_i, double* bu, double* bi);
/* One half-epoch of baseline_als (optimize_baselines.pyx:41-46 items / :48-53 users) over the segments
 * [seg_begin, seg_end) of one side's CSR: mine[s] = sum_{a in seg s} (r[a] - mu - other[idx[a]]) / (reg + |seg s|).
 * The unit of the multi-rank ALS: every ordered sum is evaluated on exactly one rank (bit-identical to the
 * single-GPU result), the caller all-gathers `mine` between the passes.  status_dev: DEVICE int, set to 1 where the
 * reference would raise ZeroDivisionError. */
int sb2_baseline_als_pass_dev(int64_t seg_begin, int64_t seg_end, const int64_t* ptr, const int32_t* idx, const double* r,
                              const double* other, double* mine, double global_mean, double reg, int* status_dev,
                              void* stream);
int sb2_baseline_sgd_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                         const double* r, double global_mean, int n_epochs, double reg, double lr, double* bu,
                         double* bi, void* stream);
int sb2_baseline_sgd(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                     const double* r, double global_mean, int n_epochs, double reg, double lr, double* bu,
                     double* bi);

/* ------------------------------------------------------------------------------------------------
 * SVD.  Replaces SVD.sgd, matrix_factorization.pyx:172-267 (hot loop :241-262).
 * pu (n_users x f) and qi (n_items x f) hold the rng.normal initialisation on entry (:233-236, made
 * on the host with numpy so that seeds agree) and the fitted factors on exit; bu / bi are outputs.
 * `global_mean` is the trainset mean; when biased == 0 it is ignored and biases stay 0 (:238, :253).
 * Update order is stratified (DSGD) and arithmetic is fp32: results are judged on held-out
 * RMSE / MAE (|diff| <= 0.005), not element-wise.
 * ------------------------------------------------------------------------------------------------ */
typedef struct sb2_sgd_params {
    int32_t n_factors;
    int32_t n_epochs;
    int32_t biased;
    int32_t reserved;
    double global_mean;
    double lr_bu, lr_bi, lr_pu, lr_qi, lr_yj;
    double reg_bu, reg_bi, reg_pu, reg_qi, reg_yj;
} sb2_sgd_params;

int sb2_svd_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                    const double* r, const sb2_sgd_params* prm, double* pu, double* qi, double* bu, double* bi,
                    void* stream);
int sb2_svd_fit(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                const double* r, const sb2_sgd_params* prm, double* pu, double* qi, double* bu, double* bi);

/* Resident-input form used by the benchmark: prepare once (stratify + upload), then run epochs with
 * everything already in HBM.  handle lifetime: create -> (reset ->) run* -> read -> destroy. */
typedef struct sb2_svd_plan sb2_svd_plan;
int sb2_svd_plan_create(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u_host,
                        const int32_t* i_host, const double* r_host, const sb2_sgd_params* prm, int with_yj,
                        sb2_svd_plan** out);
int sb2_svd_plan_reset(sb2_svd_plan* plan, const double* pu_host, const double* qi_host,
                       const double* yj_host);
/* device-pointer forms of create / reset / read (u_ptr / ui_idx: ur CSR, only read when with_yj) */
int sb2_svd_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, const sb2_sgd_params* prm, int with_yj, const int64_t* u_ptr,
                            const int32_t* ui_idx, void* stream, sb2_svd_plan** out);
int sb2_svd_plan_reset_dev(sb2_svd_plan* plan, const double* pu, const double* qi, const double* yj,
                           void* stream);
int sb2_svd_plan_read_dev(sb2_svd_plan* plan, double* pu, double* qi, double* bu, double* bi, double* yj,
                          void* stream);
int sb2_svd_plan_run(sb2_svd_plan* plan, int n_epochs, void* stream); /* async on stream */
int sb2_svd_plan_read(sb2_svd_plan* plan, double* pu, double* qi, double* bu, double* bi, double* yj);
void sb2_svd_plan_destroy(sb2_svd_plan* plan);
/* algorithmic bytes per rating update of the plan's kernel (DESIGN.md: 2*(2f+2)*4 + 12 for SVD) */
int64_t sb2_svd_plan_bytes_per_update(const sb2_svd_plan* plan);
int sb2_svd_plan_grid(const sb2_svd_plan* plan, int* n_blocks, int* n_sub);
/* Read-only layout of a plan (any pointer may be NULL): B blocks (CTAs), cluster size C (1 = no clusters), G lanes per
 * rating, CH 128-bit chunks per lane (0: 32 lanes stride the row), W lane-groups per CTA, whether the user / item
 * rows of a block are staged in shared memory, dependency-driven cells, dynamic shared memory per CTA, records of a
 * cell staged in shared memory, and the largest cell.  A plan with C > 1 always has stage_i == 1. */
int sb2_svd_plan_layout(const sb2_svd_plan* plan, int* n_blocks, int* cluster, int* lanes, int* chunks, int* n_sub,
                        int* stage_u, int* stage_i, int* dep_mode, int64_t* smem_bytes, int* rec_cap, int* max_cell);
/* Synchronises `stream` and reports whether the persistent kernel ran to completion: every wait of a CTA for a
 * neighbour CTA / rank is bounded (~6 s); if a partner was never scheduled (SMs held by another persistent kernel,
 * a dead peer rank) the launch drains and this returns SB2_ERR_CUDA instead of the GPU hanging.  The host forms
 * (sb2_svd_fit, sb2_svdpp_fit) check it themselves. */
int sb2_svd_plan_status(sb2_svd_plan* plan, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU ring (DSGD strata across ranks, one process per GPU; SURVEY.md 8e "SVD (DSGD)").  Replaces the same
 * loop, matrix_factorization.pyx:241-262 (SVD) / :466-498 (SVD++), for a trainset sharded by user.
 * Rank g of `world` owns the users u % world == g for the whole fit and, in sub-epoch E, the item super-block
 * (g + E) % world; the kernel itself hands every finished item block to rank g - 1 over NVLink (stores through the
 * peer mapping + system-scope release / acquire flags) -- ONE persistent launch per rank for a whole SVD fit.
 *   create:  every rank passes the SAME global COO (DEVICE arrays) and its (rank, world); it keeps its own ratings.
 *   connect: exchange the 64-byte handles between the processes (e.g. torch.distributed.all_gather) and pass the
 *            left (rank - 1) and right (rank + 1) neighbours' handles; or, inside one process, the plans themselves.
 *   reset:   sb2_svd_plan_reset_dev with the WHOLE initial matrices; then synchronise the ranks (any collective)
 *            before run: reset clears the mailboxes the neighbours write into.
 *   run:     sb2_svd_plan_run (SVD), or per epoch sb2_svd_ring_epoch_dev(phase 0) -> all-reduce(SUM) of `exchange`
 *            (n_items x (row_stride + 1) fp32, DEVICE) over the ranks -> sb2_svd_ring_epoch_dev(phase 1) (SVD++: the
 *            per-item sums of the y_j application span the users of all ranks).
 *   read:    sb2_svd_plan_read_dev returns the rank's OWN rows (n_users_local x f, n_items_local x f, local order:
 *            global id = rank + local * world); synchronise the ranks before reading / destroying.
 * ------------------------------------------------------------------------------------------------ */
int sb2_svd_ring_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, const sb2_sgd_params* prm, int with_yj, const int64_t* u_ptr,
                            const int32_t* ui_idx, int rank, int world, void* stream, sb2_svd_plan** out);
int sb2_svd_ring_ipc_handle(const sb2_svd_plan* plan, unsigned char* handle64);
int sb2_svd_ring_connect_ipc(sb2_svd_plan* plan, const unsigned char* left64, const unsigned char* right64);
int sb2_svd_ring_connect_local(sb2_svd_plan* plan, sb2_svd_plan* left, sb2_svd_plan* right);
int sb2_svd_ring_epoch_dev(sb2_svd_plan* plan, int phase, float* exchange, void* stream);
/* All ranks of a ring in ONE process on ONE GPU (the single-GPU tests of the ring): plans[0 .. n) are the ranks
 * 0 .. n-1 (n <= 4), connected with sb2_svd_ring_connect_local.  Kernels that wait for one another must never be
 * issued as separate launches on one GPU, so all ranks run as one launch of n x B co-resident CTAs -- the same
 * kernel body, the "peer" buffers being the other ranks' buffers in the same memory.  sb2_svd_ring_run_local: n_epochs
 * SVD epochs; sb2_svd_ring_epoch_local: phase 0 of one SVD++ epoch for every rank (exchange[g]: rank g's partial
 * sums; add them up, then call sb2_svd_ring_epoch_dev(plans[g], 1, sum) per rank). */
int sb2_svd_ring_run_local(sb2_svd_plan** plans, int n_plans, int n_epochs, void* stream);
int sb2_svd_ring_epoch_local(sb2_svd_plan** plans, int n_plans, float** exchange, void* stream);
int sb2_svd_ring_info(const sb2_svd_plan* plan, int64_t* n_users_local, int64_t* n_items_local,
                      int64_t* n_ratings_local, int* row_stride);
/* Per-CTA counters of the last run, cycles_host[n_blocks][8] (n_blocks from sb2_svd_plan_grid): SM cycles in
 * {ring wait, item-block load, rating updates, write-back, lane-group-0 updates}, then the number of
 * lane-group-0 updates, the number of waves, 0. */
int sb2_svd_plan_profile(const sb2_svd_plan* plan, int64_t* cycles_host);

/* SVD++.  Replaces SVDpp.sgd, matrix_factorization.pyx:420-504.  yj (n_items x f) in/out like qi.
 * u_ptr / ui_idx: the ur CSR (I_u).  See DESIGN.md for the per-user batching of the y_j update. */
int sb2_svdpp_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                      const double* r, const int64_t* u_ptr, const int32_t* ui_idx, const sb2_sgd_params* prm,
                      double* pu, double* qi, double* yj, double* bu, double* bi, void* stream);
int sb2_svdpp_fit(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                  const double* r, const int64_t* u_ptr, const int32_t* ui_idx, const sb2_sgd_params* prm,
                  double* pu, double* qi, double* yj, double* bu, double* bi);

/* ------------------------------------------------------------------------------------------------
 * NMF.  Replaces NMF.sgd, matrix_factorization.pyx:646-735.  Bit-exact (fp64, the reference's
 * summation order, no FMA) for biased == 0 and biased != 0.  (u, i, r) is the all_ratings COO, which
 * must be grouped by u (it is, by construction of all_ratings()).  pu / qi: rng.uniform init in,
 * factors out.  Returns SB2_ERR_ZERO_DIVISION where the reference raises (:723, :730).
 * ------------------------------------------------------------------------------------------------ */
typedef struct sb2_nmf_params {
    int32_t n_factors;
    int32_t n_epochs;
    int32_t biased;
    int32_t reserved;
    double global_mean;
    double reg_pu, reg_qi, reg_bu, reg_bi, lr_bu, lr_bi;
} sb2_nmf_params;

int sb2_nmf_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                    const double* r, const sb2_nmf_params* prm, double* pu, double* qi, double* bu, double* bi,
                    void* stream);
int sb2_nmf_fit(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                const double* r, const sb2_nmf_params* prm, double* pu, double* qi, double* bu, double* bi);

/* Epoch-at-a-time form for the multi-GPU fit (device pointers).  The plan holds what depends only on the rating
 * structure; the COO arrays are borrowed and must outlive it.  One epoch restricted to users
 * [user_begin, user_end) and items [item_begin, item_end) reads the full pu_cur / qi_cur and writes those rows
 * of pu_new / qi_new: every ordered accumulator sum is evaluated on exactly one rank, so sharded results stay
 * bit-identical; the caller all-gathers the new factors between epochs.  bu / bi (biased model) are advanced in
 * place by the sequential recursion, which every rank replays.  sb2_nmf_plan_status synchronises the stream and
 * reports SB2_ERR_ZERO_DIVISION / SB2_ERR_INVALID (input not grouped by user). */
typedef struct sb2_nmf_plan sb2_nmf_plan;
int sb2_nmf_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, int n_factors, void* stream, sb2_nmf_plan** out);
int sb2_nmf_plan_epoch_dev(sb2_nmf_plan* plan, const sb2_nmf_params* prm, const double* pu_cur, const double* qi_cur,
                           double* pu_new, double* qi_new, double* bu, double* bi, int64_t user_begin,
                           int64_t user_end, int64_t item_begin, int64_t item_end, void* stream);
int sb2_nmf_plan_status(sb2_nmf_plan* plan, void* stream);
void sb2_nmf_plan_destroy(sb2_nmf_plan* plan);

/* ------------------------------------------------------------------------------------------------
 * Batched estimate for the factor models.  Replaces SVD.estimate (matrix_factorization.pyx:269-299),
 * NMF.estimate (:737-761) and SVDpp.estimate (:506-522; yj != NULL) called once per pair by
 * AlgoBase.test (algo_base.py:191-218).  u[k] < 0 / i[k] < 0 encode an unknown user / item.
 * impossible[k] = 1 where the reference raises PredictionImpossible.
 * n_factors = 0 with biased = 1 is BaselineOnly.estimate (baseline_only.py:33-46): (mu + bu[u]) + bi[i], pu / qi unused.
 * ------------------------------------------------------------------------------------------------ */
int sb2_mf_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int n_factors, int biased,
                       double global_mean, const double* pu, const double* qi, const double* bu,
                       const double* bi, const double* yj, const int64_t* u_ptr, const int32_t* ui_idx,
                       double* est, uint8_t* impossible, void* stream);
int sb2_mf_predict(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_users, int64_t n_items,
                   int n_factors, int biased, double global_mean, const double* pu, const double* qi,
                   const double* bu, const double* bi, const double* yj, const int64_t* u_ptr,
                   const int32_t* ui_idx, double* est, uint8_t* impossible);

/* ------------------------------------------------------------------------------------------------
 * Batched k-NN estimate.  Replaces KNNBasic.estimate (knns.py:99-123) and KNNBaseline.estimate
 * (:274-309): gather sim[x, x2] over yr[y], stable top-k (heapq.nlargest semantics), ordered fp64
 * weighted sum -- bit-identical to the reference.
 * mode: 0 = KNNBasic; 1 = KNNBaseline with x = user (user_based); 2 = KNNBaseline with x = item;
 *       3 = KNNWithMeans (knns.py:178-208; bx = means[n_x], by unused); 4 = KNNWithZScore (:372-403; bx = means,
 *       by = sigmas, both indexed by x).
 * x[k] / y[k] < 0 = unknown.  actual_k[k] = -1 where the reference reports no actual_k.
 * impossible[k]: 1 = PredictionImpossible, 2 = the reference would raise ZeroDivisionError.
 * sim: n_x x n_x row-major with leading dimension sim_ld (>= n_x).
 * ------------------------------------------------------------------------------------------------ */
int sb2_knn_predict_dev(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, const double* sim,
                        int64_t sim_ld, const int64_t* y_ptr, const int32_t* x_idx, const double* r, int k,
                        int min_k, int mode, double global_mean, const double* bx, const double* by,
                        double* est, int32_t* actual_k, uint8_t* impossible, void* stream);
int sb2_knn_predict(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, int64_t n_y,
                    const double* sim, const int64_t* y_ptr, const int32_t* x_idx, const double* r, int k,
                    int min_k, int mode, double global_mean, const double* bx, const double* by, double* est,
                    int32_t* actual_k, uint8_t* impossible);
/* The same estimates from a block of similarity rows: pair k reads sim[x[k], .] at sim + sim_row[k] * sim_ld
 * (for known pairs).  bx, by, the neighbour ids and every other array stay indexed by the global x / y.
 * sb2_knn_predict_dev is this call with sim_row = x. */
int sb2_knn_predict_rows_dev(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, const double* sim,
                             int64_t sim_ld, const int32_t* sim_row, const int64_t* y_ptr, const int32_t* x_idx,
                             const double* r, int k, int min_k, int mode, double global_mean, const double* bx,
                             const double* by, double* est, int32_t* actual_k, uint8_t* impossible, void* stream);

/* ------------------------------------------------------------------------------------------------
 * SlopeOne ("next" row 4 of the hot-path table).  sb2_slope_one_fit replaces the two loops of
 * SlopeOne.fit (prediction_algorithms/slope_one.pyx:59-70): freq[i][j] = number of users who rated both
 * items (n_items x n_items int64; diagonal = raters of i), dev[i][j] = mean over those users of
 * r_ui - r_uj with the ratings TRUNCATED to C ints exactly as the reference's `cdef int r_ui, r_uj` does
 * (slope_one.pyx:52); 0 / 0 = NaN where freq is 0; dev[j][i] = -dev[i][j]; dev[i][i] = 0.  Both are
 * by-products of the similarity contractions (freq = M M^T, sum r_ui = R M^T) on the tensor cores and are
 * bit-identical to the reference.  u_ptr / i_idx / r: the ur CSR (trainset.ur flattened, user-major).
 * sb2_slope_one_predict replaces SlopeOne.estimate (:82-97); user_mean[u] is computed by the host mirror.
 * impossible[k] = 1 where the reference raises PredictionImpossible (u[k] < 0 or i[k] < 0).
 * ------------------------------------------------------------------------------------------------ */
int sb2_slope_one_fit_dev(int64_t n_items, int64_t n_users, const int64_t* u_ptr, const int32_t* i_idx,
                          const double* r, int64_t nnz, int64_t* freq_out, double* dev_out, void* stream);
int sb2_slope_one_fit(int64_t n_items, int64_t n_users, const int64_t* u_ptr, const int32_t* i_idx,
                      const double* r, int64_t* freq_out, double* dev_out);
int sb2_slope_one_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_items,
                              const int64_t* freq, const double* dev, const int64_t* u_ptr, const int32_t* i_idx,
                              const double* user_mean, double* est, uint8_t* impossible, void* stream);

/* ------------------------------------------------------------------------------------------------
 * CoClustering.  sb2_coclustering_fit replaces CoClustering.fit's epoch loop and compute_averages
 * (prediction_algorithms/co_clustering.pyx:68-155, :157-237): n_epochs x (averages, user pass, item pass),
 * then the final averages.  Bit-identical to the reference: ratings are truncated to C ints like its
 * `cdef int r`; the cluster averages are exact integer sums / counts (global_mean for an empty cluster); every
 * errors[c] is an ordered fp64 sum in ur[u] (ir[i]) list order; argmin takes the first minimum.
 * u_ptr / ui_idx / u_r: the ur CSR; i_ptr / iu_idx / i_r: the ir CSR (nnz entries each).
 * user_mean / item_mean: np.mean of each ur[u] / ir[i] list (computed by the caller, untruncated).
 * cltr_u[n_users], cltr_i[n_items] (int32, in/out): the rng.randint draw on entry, the final clusters on exit.
 * avg_cltr_u[n_cltr_u], avg_cltr_i[n_cltr_i], avg_cocltr[n_cltr_u x n_cltr_i] (row-major): outputs.
 * SB2_ERR_INVALID for n_cltr_u < 1 or n_cltr_i < 1, an initial cluster out of range, or a rating outside the C
 * int range (the reference raises OverflowError).  The _dev form enqueues the whole fit and synchronises
 * `stream` once at the end to read that status.
 * sb2_coclustering_predict_dev replaces CoClustering.estimate (co_clustering.pyx, after compute_averages):
 * u[k] < 0 or i[k] < 0 (unknown) gives global_mean -- an estimate, not PredictionImpossible.
 * ------------------------------------------------------------------------------------------------ */
int sb2_coclustering_fit_dev(int64_t n_users, int64_t n_items, int64_t nnz, const int64_t* u_ptr,
                             const int32_t* ui_idx, const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx,
                             const double* i_r, const double* user_mean, const double* item_mean,
                             double global_mean, int n_cltr_u, int n_cltr_i, int n_epochs, int32_t* cltr_u,
                             int32_t* cltr_i, double* avg_cltr_u, double* avg_cltr_i, double* avg_cocltr,
                             void* stream);
int sb2_coclustering_fit(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx,
                         const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                         const double* user_mean, const double* item_mean, double global_mean, int n_cltr_u,
                         int n_cltr_i, int n_epochs, int32_t* cltr_u, int32_t* cltr_i, double* avg_cltr_u,
                         double* avg_cltr_i, double* avg_cocltr);
int sb2_coclustering_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_users,
                                 int64_t n_items, int n_cltr_i, const int32_t* cltr_u, const int32_t* cltr_i,
                                 const double* user_mean, const double* item_mean, const double* avg_cltr_u,
                                 const double* avg_cltr_i, const double* avg_cocltr, double global_mean,
                                 double* est, void* stream);

/* ------------------------------------------------------------------------------------------------
 * AlgoBase.get_neighbors (algo_base.py:303-334) on the device-resident similarity matrix: for each
 * requested row x = rows[b], the k other ids with the largest sim[x, .], in the order of the reference's
 * stable descending sort (ties by ascending id).  out: n_rows x k int32, padded with -1 when fewer than
 * k other ids exist (the reference returns a shorter list) or rows[b] is out of range.
 * ------------------------------------------------------------------------------------------------ */
int sb2_get_neighbors_dev(int64_t n_x, const double* sim, int64_t sim_ld, int64_t n_rows, const int32_t* rows,
                          int k, int32_t* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Top-N recommendations (AlgoBase.get_top_n / top_n_inner): the FAQ's get_top_n over
 * algo.test(trainset.build_anti_testset()), on the device.
 * sb2_mf_score_block_dev: scores[b * ld + i] = the estimate sb2_mf_predict_dev returns for the pair
 * (rows[b], i), bit for bit, for every b < n_rows and every item i < n_items (SVD, SVD++ with yj / u_ptr /
 * ui_idx, NMF, and BaselineOnly with f = 0, pu = qi = NULL).  rows[b] must be known users (0 <= rows[b] <
 * n_users); biased as in sb2_mf_predict_dev.  Three launches per call (factor repacks, then the scorer).
 * sb2_top_n_select_dev: for each row b, the candidates are the items rows[b] did not rate (ur CSR u_ptr /
 * ui_idx).  Each gets the value AlgoBase.test gives it: scores[b * ld + i], replaced by default_est where
 * impossible[b * ld + i] == 1 (impossible may be NULL: no impossible pairs), minus offset, then
 * min(high, .) and max(low, .).  Output: the first n candidates in (value desc, item asc) order -- Python's
 * stable sort(reverse=True) of the anti-testset -- with -0.0 equal to +0.0 and NaN after every number:
 * items_out[b * n + j] (int32 inner ids) and est_out[b * n + j] (the values), padded with -1 / NaN;
 * count_out[b] = the number emitted.  One launch per call; one pass over each row for n <= 2048 and one
 * more per further 2048 entries.  SB2_ERR_INVALID for n < 1; SB2_ERR_ZERO_DIVISION where a candidate has
 * impossible == 2 (the reference raises ZeroDivisionError; the call then synchronises `stream` to read
 * that status); SB2_ERR_UNSUPPORTED when the rated-item bitmap (n_items bits) does not fit in shared memory
 * (about 1.4 M items).
 * ------------------------------------------------------------------------------------------------ */
int sb2_mf_score_block_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, int f, int biased,
                           double global_mean, const double* pu, const double* qi, const double* bu,
                           const double* bi, const double* yj, const int64_t* u_ptr, const int32_t* ui_idx,
                           double* scores, int64_t ld, void* stream);
int sb2_top_n_select_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                         const uint8_t* impossible, double default_est, double offset, double low, double high,
                         const int64_t* u_ptr, const int32_t* ui_idx, int n, int32_t* items_out,
                         double* est_out, int32_t* count_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Per-user counts behind accuracy.fcp and accuracy.precision_recall_at_k (DESIGN.md section 3.7).  All
 * arrays are DEVICE arrays.  The n predictions are grouped into n_seg segments (users): segment s holds
 * entries [seg_ptr[s], seg_ptr[s + 1]) of r (true ratings) and est (estimates), in prediction order;
 * seg_ptr (int64, n_seg + 1 entries) must start at 0, not decrease and end at n, else SB2_ERR_INVALID.
 * Compares are fp64 (NaN compares false, -0.0 == +0.0).  i and j run over one segment, i == j included.
 * sb2_fcp_counts_dev: counts[2 s] = #{(i, j) : est_i > est_j and r_i > r_j},
 *   counts[2 s + 1] = #{(i, j) : est_i >= est_j and r_i < r_j}.
 * sb2_precision_at_k_counts_dev: with m = the segment's length, rank_j = #{i : est_i > est_j} +
 *   #{i < j : est_i == est_j} (Python's stable sort(reverse=True)) and top = {j : rank_j < k_eff[s]}
 *   (k_eff int64 per segment; k_eff >= m: every entry, k_eff <= 0: none):
 *   counts[3 s] = #{j : r_j >= threshold}, counts[3 s + 1] = #{j in top : est_j >= threshold},
 *   counts[3 s + 2] = #{j in top : r_j >= threshold and est_j >= threshold}.
 * counts: int64, zeroed by the call.  One launch per call; the call synchronises `stream` to check the
 * offsets, so the counts are ready when it returns.
 * ------------------------------------------------------------------------------------------------ */
int sb2_fcp_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r, const double* est,
                       int64_t* counts, void* stream);
int sb2_precision_at_k_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r,
                                  const double* est, const int64_t* k_eff, double threshold, int64_t* counts,
                                  void* stream);

/* ------------------------------------------------------------------------------------------------
 * Hits of top-N lists against held-out relevant items (AlgoBase.top_n_measures; the definition is
 * accuracy.top_n_measures, DESIGN.md section 3.9).  All arrays are DEVICE arrays.  items (int32, row b at
 * items + b * ld) and count (int32 per row) are a block of sb2_top_n_select_dev's output; w <= ld is the
 * cutoff.  Row b's relevant items are rel_idx[rel_ptr[b], rel_ptr[b + 1]) (rel_ptr int64, n_rows + 1
 * entries, offsets into rel_idx of rel_len entries), distinct inner item ids in strictly ascending order.
 * With H_b = {p < min(count[b], w) : items[b * ld + p] in row b's list}:
 *   hits[b] = |H_b|, rr[b] = the sum of inv[p] over H_b, dcg[b] = the sum of disc[p] over H_b,
 * each sum taken in ascending p from +0.0 with one fp64 add per term (no FMA).  inv and disc (fp64, at least w
 * entries) are the host's tables, so no logarithm is evaluated on the device.  SB2_ERR_INVALID for a null
 * pointer, w < 0, ld < w, or offsets outside [0, rel_len], decreasing, or a list not strictly ascending (checked
 * inside the kernel).  One launch per call; the call synchronises `stream` to read that check.
 * ------------------------------------------------------------------------------------------------ */
int sb2_top_n_hits_dev(int64_t n_rows, const int32_t* items, int64_t ld, const int32_t* count, int w,
                       const int64_t* rel_ptr, const int32_t* rel_idx, int64_t rel_len, const double* inv,
                       const double* disc, int32_t* hits, double* rr, double* dcg, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Coverage, novelty and intra-list similarity of top-N lists (AlgoBase.top_n_list_measures; the definition is
 * accuracy.top_n_list_measures, DESIGN.md section 3.11).  All arrays are DEVICE arrays.  items (int32, row b at
 * items + b * ld), est (fp64, same layout) and count (int32 per row) are a block of sb2_top_n_select_dev's output;
 * w <= ld is the cutoff.  With c_b = min(count[b], w) and L_b = items[b * ld + 0 .. c_b):
 *   covered[b] = 1 when some p < c_b has est[b * ld + p] >= threshold (when has_threshold is 0: when c_b > 0), else 0;
 *   nov[b] = the sum of info[L_b[p]] over p ascending;
 *   ils[b] = the sum of sim[L_b[p] * n_items + L_b[q]] over p < q, p ascending and q ascending inside it (only when
 *   sim is not null; sim is the n_items x n_items row-major item-item similarity);
 *   seen[L_b[p]] = 1 for every p (a byte per item; the call never clears it, so one zeroed array can collect several
 *   calls).
 * Each sum is taken from +0.0 with one fp64 add per term (no FMA).  info (fp64, n_items entries) is the host's
 * self-information table, so no logarithm is evaluated on the device.  est may be null when has_threshold is 0.
 * SB2_ERR_INVALID for a null pointer, w < 0, ld < w, or a listed item outside [0, n_items) (checked inside the kernel;
 * such an item is read nowhere).  One launch per call; the call synchronises `stream` to read that check.
 * ------------------------------------------------------------------------------------------------ */
int sb2_top_n_lists_dev(int64_t n_rows, const int32_t* items, int64_t ld, const double* est, const int32_t* count,
                        int w, int has_threshold, double threshold, int64_t n_items, const double* info,
                        const double* sim, int32_t* covered, double* nov, double* ils, uint8_t* seen, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Where held-out items land in each user's full ranking (AlgoBase.rank_measures: AUC, MRR, MPR; the definition is
 * accuracy.rank_measures, DESIGN.md section 3.12).  All arrays are DEVICE arrays.  rows, scores / ld, impossible,
 * default_est, offset, low, high and the ur CSR u_ptr / ui_idx are exactly sb2_top_n_select_dev's: the candidates
 * of row b are the items rows[b] did not rate, ranked in that function's order.  rel_idx[rel_ptr[b] ..
 * rel_ptr[b + 1]) (int64 offsets into rel_idx, rel_len entries) are row b's relevant inner item ids, strictly
 * ascending; a relevant item the user rated is no candidate.  With the position of a candidate = the number of
 * candidates ranked before it, for every row b:
 *   c[b] = the number of candidates, k[b] = the number of relevant candidates, s[b] (int64) = the sum of their
 *   positions, f[b] = the smallest of them, or -1 when k[b] == 0.
 * SB2_ERR_INVALID for a null pointer, ld < n_items, or a row whose offsets leave [0, rel_len], decrease, or whose
 * list is not strictly ascending inside [0, n_items) (checked inside the kernel; such a row's outputs are not
 * written); SB2_ERR_ZERO_DIVISION where a candidate has impossible == 2, as sb2_top_n_select_dev;
 * SB2_ERR_UNSUPPORTED when the rated-item bitmap does not fit in shared memory (about 1.4 M items).  One launch per
 * call, one pass over each row's scores per 2048 relevant candidates (at least one); the call synchronises `stream`
 * to read its checks.
 * ------------------------------------------------------------------------------------------------ */
int sb2_top_n_ranks_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                        const uint8_t* impossible, double default_est, double offset, double low, double high,
                        const int64_t* u_ptr, const int32_t* ui_idx, const int64_t* rel_ptr, const int32_t* rel_idx,
                        int64_t rel_len, int32_t* c, int32_t* k, int64_t* s, int32_t* f, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Row shard of a SYMMETRIC multi-rank similarity build (SURVEY.md 8e "cyclic upper-triangular tile sharding").
 * Same arguments as sb2_sim_build_dev, but only sim[i][j] with row_begin <= i < row_end and j >= row_begin is
 * computed (tiles at or above the block diagonal; the shard's own diagonal square is mirrored like the
 * reference mirrors, similarities.pyx:95).  Columns j < row_begin of sim_out are left untouched: they are
 * the transposes of blocks computed by the shards before this one (surprise_b200/distributed.py exchanges
 * them over NCCL).  With row ranges of equal triangular area every rank does 1/N of the single-GPU work.
 * ------------------------------------------------------------------------------------------------ */
int sb2_sim_build_upper_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx,
                            const double* r, int64_t nnz, int rating_denom, int min_support, double global_mean,
                            const double* x_biases, const double* y_biases, double shrinkage, int64_t row_begin,
                            int64_t row_end, double* sim_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * rating_denom for sb2_sim_build*: the smallest d in {1, 2, 4, 5, 10, 20, 100, 1000} such that every rating
 * (DEVICE array) is an integer multiple of 1/d within [0, 65535/d] (relative tolerance 1e-9, the same test
 * sb2_sim_build applies); *denom_out (HOST int) = 0 when the ratings lie on none of these grids.
 * ------------------------------------------------------------------------------------------------ */
int sb2_rating_denominator_dev(const double* r, int64_t nnz, int* denom_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Listed rows of the similarity matrix, for k-NN models whose n_x x n_x matrix is not kept: out[b * ld + j] =
 * sim[rows[b]][j] for b < n_rows and every j < n_x, bit for bit the same rows of sb2_sim_build_dev(0, n_x) --
 * entries left of the diagonal included, evaluated as the pair (min, max) the way the reference mirrors them
 * (similarities.pyx:95).  Same arguments and statuses as sb2_sim_build_dev (SB2_ERR_ZERO_DIVISION for msd, duplicated
 * pairs on the general path); rows (DEVICE int32) may come in any order and repeat; a row outside [0, n_x) is
 * SB2_ERR_INVALID; ld >= n_x.  The tensor path packs the A side from the listed rows and contracts them against all
 * n_x rows (2 G n_rows n_x n_y operations, no symmetry); the general path runs the listed rows' co-ratings.  The path
 * is chosen by the cost model for n_rows where both paths give the same bits (cosine / msd / pearson on a power-of-two
 * rating grid), otherwise as the full build chooses it.  Synchronises `stream`.
 * ------------------------------------------------------------------------------------------------ */
int sb2_sim_build_rows_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx,
                           const double* r, int64_t nnz, int rating_denom, int min_support, double global_mean,
                           const double* x_biases, const double* y_biases, double shrinkage, const int32_t* rows,
                           int64_t n_rows, double* out, int64_t ld, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SURPRISE_B200_H */
