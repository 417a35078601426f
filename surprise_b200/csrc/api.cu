// extern "C" boundary of libsurprise_b200.so (declared in include/surprise_b200.h).
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "sim_gemm.cuh"

struct sb2_svd_plan;
struct sb2_nmf_plan;

namespace sb2 {

static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int64_t& launch_counter() { return g_launches; }

int sm_count() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
            n = 0;
    }
    return n > 0 ? n : 1;
}

// implemented in the other translation units
int sim_build_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                  int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                  const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end, double* sim_out,
                  cudaStream_t st);
int sim_build_upper_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                        int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                        const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end, double* sim_out,
                        cudaStream_t st);
int sim_build_rows_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                       int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                       const double* y_biases, double shrinkage, const int32_t* rows, int64_t n_rows, double* out,
                       int64_t ld, cudaStream_t st);
int rating_denominator_dev(const double* r, int64_t nnz, int* denom_out, cudaStream_t st);
int baseline_als_dev(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx, const double* u_r,
                     const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r, double mu, int n_epochs,
                     double reg_u, double reg_i, double* bu, double* bi, cudaStream_t st);
int baseline_als_pass_dev(int64_t seg_begin, int64_t seg_end, const int64_t* ptr, const int32_t* idx, const double* r,
                          const double* other, double* mine, double mu, double reg, int* status_dev, cudaStream_t st);
int baseline_sgd_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                     double mu, int n_epochs, double reg, double lr, double* bu, double* bi, cudaStream_t st);
int nmf_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                const sb2_nmf_params* prm, double* pu, double* qi, double* bu, double* bi, cudaStream_t st);
int nmf_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                        int n_factors, cudaStream_t st, sb2_nmf_plan** out);
int nmf_plan_epoch_dev(sb2_nmf_plan* p, const sb2_nmf_params* prm, const double* pu_cur, const double* qi_cur,
                       double* pu_new, double* qi_new, double* bu, double* bi, int64_t u0, int64_t u1, int64_t i0,
                       int64_t i1, cudaStream_t st);
int nmf_plan_status(sb2_nmf_plan* p, cudaStream_t st);
void nmf_plan_destroy(sb2_nmf_plan* p);
int mf_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int f, int biased, double mu, const double* pu,
                   const double* qi, const double* bu, const double* bi, const double* yj, const int64_t* u_ptr,
                   const int32_t* ui_idx, double* est, uint8_t* impossible, cudaStream_t st);
int knn_predict_dev(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, const double* sim,
                    int64_t sim_ld, const int32_t* sim_row, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                    int k, int min_k, int mode, double mu, const double* bx, const double* by, double* est,
                    int32_t* actual_k, uint8_t* impossible, cudaStream_t st);
int get_neighbors_dev(int64_t n_x, const double* sim, int64_t sim_ld, int64_t n_rows, const int32_t* rows, int k,
                      int32_t* out, cudaStream_t st);
int slope_one_fit_dev(int64_t n_items, int64_t n_users, const int64_t* u_ptr, const int32_t* i_idx, const double* r,
                      int64_t nnz, int64_t* freq_out, double* dev_out, cudaStream_t st);
int slope_one_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_items, const int64_t* freq,
                          const double* dev, const int64_t* u_ptr, const int32_t* i_idx, const double* user_mean,
                          double* est, uint8_t* impossible, cudaStream_t st);
int coclustering_fit_dev(int64_t n_users, int64_t n_items, int64_t nnz, const int64_t* u_ptr, const int32_t* ui_idx,
                         const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                         const double* user_mean, const double* item_mean, double mu, int n_cu, int n_ci, int n_epochs,
                         int32_t* cltr_u, int32_t* cltr_i, double* avg_u, double* avg_i, double* avg_co,
                         cudaStream_t st);
int coclustering_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_users, int64_t n_items,
                             int n_ci, const int32_t* cltr_u, const int32_t* cltr_i, const double* user_mean,
                             const double* item_mean, const double* avg_u, const double* avg_i, const double* avg_co,
                             double mu, double* est, cudaStream_t st);
int mf_score_block_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, int f, int biased, double mu,
                       const double* pu, const double* qi, const double* bu, const double* bi, const double* yj,
                       const int64_t* u_ptr, const int32_t* ui_idx, double* scores, int64_t ld, cudaStream_t st);
int top_n_select_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                     const uint8_t* impossible, double default_est, double offset, double low, double high,
                     const int64_t* u_ptr, const int32_t* ui_idx, int n, int32_t* items_out, double* est_out,
                     int32_t* count_out, cudaStream_t st);
int fcp_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r, const double* est,
                   int64_t* counts, cudaStream_t st);
int precision_at_k_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r, const double* est,
                              const int64_t* k_eff, double threshold, int64_t* counts, cudaStream_t st);
int top_n_hits_dev(int64_t n_rows, const int32_t* items, int64_t ld, const int32_t* count, int w,
                   const int64_t* rel_ptr, const int32_t* rel_idx, int64_t rel_len, const double* inv,
                   const double* disc, int32_t* hits, double* rr, double* dcg, cudaStream_t st);
int top_n_lists_dev(int64_t n_rows, const int32_t* items, int64_t ld, const double* est, const int32_t* count, int w,
                    int has_threshold, double threshold, int64_t n_items, const double* info, const double* sim,
                    int32_t* covered, double* nov, double* ils, uint8_t* seen, cudaStream_t st);
int top_n_ranks_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                    const uint8_t* impossible, double default_est, double offset, double low, double high,
                    const int64_t* u_ptr, const int32_t* ui_idx, const int64_t* rel_ptr, const int32_t* rel_idx,
                    int64_t rel_len, int32_t* c, int32_t* k, int64_t* s, int32_t* f, cudaStream_t st);
int svd_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                        const double* r, const sb2_sgd_params* prm, int with_yj, const int64_t* u_ptr,
                        const int32_t* ui_idx, int rank, int world, cudaStream_t st, sb2_svd_plan** out);
int svd_plan_reset_dev(sb2_svd_plan* p, const double* pu0, const double* qi0, const double* yj0, cudaStream_t st);
int svd_plan_run(sb2_svd_plan* p, int n_epochs, cudaStream_t st);
int svd_plan_read_dev(sb2_svd_plan* p, double* pu, double* qi, double* bu, double* bi, double* yj, cudaStream_t st);
void svd_plan_destroy(sb2_svd_plan* p);
int64_t svd_plan_bytes_per_update(const sb2_svd_plan* p);
void svd_plan_grid(const sb2_svd_plan* p, int* b, int* w);
void svd_plan_layout(const sb2_svd_plan* p, int* b, int* c, int* g, int* ch, int* w, int* stage_u, int* stage_i,
                     int* dep_mode, int64_t* smem, int* rec_cap, int* max_cell);
int svd_plan_status(sb2_svd_plan* p, cudaStream_t st);
int svd_ring_epoch_dev(sb2_svd_plan* p, int phase, float* xch, cudaStream_t st);
int svd_ring_run_local(sb2_svd_plan** plans, int n, int n_epochs, cudaStream_t st);
int svd_ring_epoch_local(sb2_svd_plan** plans, int n, float** xch, cudaStream_t st);
int svd_ring_ipc_handle(const sb2_svd_plan* p, unsigned char* out64);
int svd_ring_connect_ipc(sb2_svd_plan* p, const unsigned char* left64, const unsigned char* right64);
int svd_ring_connect_local(sb2_svd_plan* p, sb2_svd_plan* left, sb2_svd_plan* right);
void svd_ring_info(const sb2_svd_plan* p, int64_t* nu_loc, int64_t* ni_loc, int64_t* n_loc, int* stride);
int svd_plan_profile(const sb2_svd_plan* p, long long* out_host);
void svd_plan_dims(const sb2_svd_plan* p, int64_t* n_users, int64_t* n_items, int* f, int* with_yj);

static int ensure_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        set_error("no usable CUDA device (%s): surprise_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        cudaGetLastError();
        return SB2_ERR_CUDA;
    }
    // Keep stream-ordered allocations cached in the device's default pool instead of returning them to
    // the OS at every synchronisation (the default release threshold is 0): the similarity path allocates
    // GBs of panels / planes per call and re-mapping them would dwarf the kernels.
    static thread_local int pool_ready_dev = -1;
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && dev != pool_ready_dev) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
            uint64_t thr = UINT64_MAX;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
        pool_ready_dev = dev;
    }
    return SB2_OK;
}

template <class T>
static int download(T* host, const void* dev, size_t n, cudaStream_t st) {
    if (n) SB2_CUDA(cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, st));
    return SB2_OK;
}

}  // namespace sb2

using namespace sb2;

extern "C" {

const char* sb2_last_error(void) { return g_err; }
int sb2_version(void) { return 100; }
int64_t sb2_launch_count(void) { return g_launches; }
void sb2_reset_launch_count(void) { g_launches = 0; }

int sb2_device_info(int* sm, int* cc_major, int* cc_minor, int64_t* total_mem) {
    SB2_TRY(ensure_device());
    int dev = 0;
    SB2_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    SB2_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm) *sm = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem) *total_mem = (int64_t)p.totalGlobalMem;
    return SB2_OK;
}

// ---- similarities ------------------------------------------------------------------------------
int sb2_sim_build_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                      int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                      const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end, double* sim_out,
                      void* stream) {
    SB2_TRY(ensure_device());
    return sim_build_dev(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases,
                         y_biases, shrinkage, row_begin, row_end, sim_out, (cudaStream_t)stream);
}

int sb2_sim_build(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                  int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                  const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end, double* sim_out) {
    SB2_TRY(ensure_device());
    if (n_x <= 0 || row_end <= row_begin) {
        set_error("sim_build: invalid argument");
        return SB2_ERR_INVALID;
    }
    cudaStream_t st = nullptr;
    DevBuf d_ptr, d_idx, d_r, d_bx, d_by, d_sim;
    SB2_TRY(upload(d_ptr, y_ptr, (size_t)n_y + 1, st));
    SB2_TRY(upload(d_idx, x_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_r, r, (size_t)nnz, st));
    if (kind == SB2_SIM_PEARSON_BASELINE) {
        if (!x_biases || !y_biases) {
            set_error("sim_build: pearson_baseline needs x_biases and y_biases");
            return SB2_ERR_INVALID;
        }
        SB2_TRY(upload(d_bx, x_biases, (size_t)n_x, st));
        SB2_TRY(upload(d_by, y_biases, (size_t)n_y, st));
    }
    const size_t out_elems = (size_t)(row_end - row_begin) * (size_t)n_x;
    SB2_TRY(d_sim.alloc(out_elems * sizeof(double), st));
    SB2_TRY(sim_build_dev(kind, n_x, n_y, d_ptr.as<int64_t>(), d_idx.as<int32_t>(), d_r.as<double>(), nnz, rating_denom,
                          min_support, global_mean, d_bx.as<double>(), d_by.as<double>(), shrinkage, row_begin, row_end,
                          d_sim.as<double>(), st));
    SB2_TRY(download(sim_out, d_sim.p, out_elems, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_gemm_u8_selftest_dev(int use_tc, int64_t m, int64_t n, int64_t k, const uint8_t* a, const uint8_t* b,
                             int32_t* c, void* stream) {
    SB2_TRY(ensure_device());
    return gemm_u8_selftest(use_tc, m, n, k, a, b, c, (cudaStream_t)stream);
}

// ---- baselines ---------------------------------------------------------------------------------
int sb2_baseline_als_dev(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx,
                         const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                         double global_mean, int n_epochs, double reg_u, double reg_i, double* bu, double* bi,
                         void* stream) {
    SB2_TRY(ensure_device());
    return baseline_als_dev(n_users, n_items, u_ptr, ui_idx, u_r, i_ptr, iu_idx, i_r, global_mean, n_epochs, reg_u,
                            reg_i, bu, bi, (cudaStream_t)stream);
}

int sb2_baseline_als(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx, const double* u_r,
                     const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r, double global_mean, int n_epochs,
                     double reg_u, double reg_i, double* bu, double* bi) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    // nnz is the last CSR offset
    const int64_t nnz = u_ptr[n_users];
    DevBuf d_up, d_ui, d_ur, d_ip, d_iu, d_ir, d_bu, d_bi;
    SB2_TRY(upload(d_up, u_ptr, (size_t)n_users + 1, st));
    SB2_TRY(upload(d_ui, ui_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_ur, u_r, (size_t)nnz, st));
    SB2_TRY(upload(d_ip, i_ptr, (size_t)n_items + 1, st));
    SB2_TRY(upload(d_iu, iu_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_ir, i_r, (size_t)nnz, st));
    SB2_TRY(d_bu.alloc((size_t)n_users * 8, st));
    SB2_TRY(d_bi.alloc((size_t)n_items * 8, st));
    SB2_TRY(baseline_als_dev(n_users, n_items, d_up.as<int64_t>(), d_ui.as<int32_t>(), d_ur.as<double>(),
                             d_ip.as<int64_t>(), d_iu.as<int32_t>(), d_ir.as<double>(), global_mean, n_epochs, reg_u,
                             reg_i, d_bu.as<double>(), d_bi.as<double>(), st));
    SB2_TRY(download(bu, d_bu.p, (size_t)n_users, st));
    SB2_TRY(download(bi, d_bi.p, (size_t)n_items, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_baseline_als_pass_dev(int64_t seg_begin, int64_t seg_end, const int64_t* ptr, const int32_t* idx, const double* r,
                              const double* other, double* mine, double global_mean, double reg, int* status_dev,
                              void* stream) {
    SB2_TRY(ensure_device());
    if (!ptr || !idx || !r || !other || !mine || !status_dev || seg_begin < 0) {
        set_error("baseline_als_pass: invalid argument");
        return SB2_ERR_INVALID;
    }
    return baseline_als_pass_dev(seg_begin, seg_end, ptr, idx, r, other, mine, global_mean, reg, status_dev,
                                 (cudaStream_t)stream);
}

int sb2_baseline_sgd_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                         const double* r, double global_mean, int n_epochs, double reg, double lr, double* bu,
                         double* bi, void* stream) {
    SB2_TRY(ensure_device());
    return baseline_sgd_dev(n_users, n_items, n, u, i, r, global_mean, n_epochs, reg, lr, bu, bi,
                            (cudaStream_t)stream);
}

int sb2_baseline_sgd(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                     double global_mean, int n_epochs, double reg, double lr, double* bu, double* bi) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    DevBuf d_u, d_i, d_r, d_bu, d_bi;
    SB2_TRY(upload(d_u, u, (size_t)n, st));
    SB2_TRY(upload(d_i, i, (size_t)n, st));
    SB2_TRY(upload(d_r, r, (size_t)n, st));
    SB2_TRY(d_bu.alloc((size_t)n_users * 8, st));
    SB2_TRY(d_bi.alloc((size_t)n_items * 8, st));
    SB2_TRY(baseline_sgd_dev(n_users, n_items, n, d_u.as<int32_t>(), d_i.as<int32_t>(), d_r.as<double>(), global_mean,
                             n_epochs, reg, lr, d_bu.as<double>(), d_bi.as<double>(), st));
    SB2_TRY(download(bu, d_bu.p, (size_t)n_users, st));
    SB2_TRY(download(bi, d_bi.p, (size_t)n_items, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

// ---- SVD / SVD++ -------------------------------------------------------------------------------
// reset -> run -> read -> status on an existing plan; destroys the plan
static int svd_like_run_plan(sb2_svd_plan* plan, const sb2_sgd_params* prm, double* pu, double* qi, double* yj, double* bu,
                             double* bi, cudaStream_t st) {
    int rc = svd_plan_reset_dev(plan, pu, qi, yj, st);
    if (rc == SB2_OK) rc = svd_plan_run(plan, prm->n_epochs, st);
    if (rc == SB2_OK) rc = svd_plan_read_dev(plan, pu, qi, bu, bi, yj, st);
    if (rc == SB2_OK) rc = svd_plan_status(plan, st);  // synchronises; a wait that hit its deadline is an error
    if (rc == SB2_OK && cudaGetLastError() != cudaSuccess) {
        set_error("svd_fit: CUDA error after the fit");
        rc = SB2_ERR_CUDA;
    }
    svd_plan_destroy(plan);
    return rc;
}

static int svd_like_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, const int64_t* u_ptr, const int32_t* ui_idx, const sb2_sgd_params* prm,
                            double* pu, double* qi, double* yj, double* bu, double* bi, cudaStream_t st) {
    sb2_svd_plan* plan = nullptr;
    SB2_TRY(svd_plan_create_dev(n_users, n_items, n, u, i, r, prm, yj != nullptr, u_ptr, ui_idx, 0, 1, st, &plan));
    return svd_like_run_plan(plan, prm, pu, qi, yj, bu, bi, st);
}

int sb2_svd_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                    const sb2_sgd_params* prm, double* pu, double* qi, double* bu, double* bi, void* stream) {
    SB2_TRY(ensure_device());
    return svd_like_fit_dev(n_users, n_items, n, u, i, r, nullptr, nullptr, prm, pu, qi, nullptr, bu, bi,
                            (cudaStream_t)stream);
}

int sb2_svdpp_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                      const int64_t* u_ptr, const int32_t* ui_idx, const sb2_sgd_params* prm, double* pu, double* qi,
                      double* yj, double* bu, double* bi, void* stream) {
    SB2_TRY(ensure_device());
    if (!yj || !u_ptr || !ui_idx) {
        set_error("svdpp_fit: yj, u_ptr and ui_idx are required");
        return SB2_ERR_INVALID;
    }
    return svd_like_fit_dev(n_users, n_items, n, u, i, r, u_ptr, ui_idx, prm, pu, qi, yj, bu, bi,
                            (cudaStream_t)stream);
}

static int svd_like_fit_host(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                             const double* r, const int64_t* u_ptr, const int32_t* ui_idx, const sb2_sgd_params* prm,
                             double* pu, double* qi, double* yj, double* bu, double* bi) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    const size_t f = (size_t)prm->n_factors;
    DevBuf d_u, d_i, d_r, d_up, d_ui, d_pu, d_qi, d_yj, d_bu, d_bi;
    SB2_TRY(upload(d_u, u, (size_t)n, st));
    SB2_TRY(upload(d_i, i, (size_t)n, st));
    SB2_TRY(upload(d_r, r, (size_t)n, st));
    if (yj) {
        SB2_TRY(upload(d_up, u_ptr, (size_t)n_users + 1, st));
        SB2_TRY(upload(d_ui, ui_idx, (size_t)n, st));
    }
    // The initial factors are not needed before the plan exists: they travel on a second stream while the ratings
    // are stratified and coloured (plan creation: ~0.1 ms of kernels + one status read-back at the ml-1M shape)
    struct Side { cudaStream_t s = nullptr; cudaEvent_t alloc = nullptr, up = nullptr; };
    static Side sides[64];   // one per device, created on first use (the host forms are not re-entrant per device)
    int dev = 0;
    SB2_CUDA(cudaGetDevice(&dev));
    Side& sd = sides[dev & 63];
    if (!sd.s) {
        SB2_CUDA(cudaStreamCreateWithFlags(&sd.s, cudaStreamNonBlocking));
        SB2_CUDA(cudaEventCreateWithFlags(&sd.alloc, cudaEventDisableTiming));
        SB2_CUDA(cudaEventCreateWithFlags(&sd.up, cudaEventDisableTiming));
    }
    cudaStream_t side = sd.s;
    cudaEvent_t ev_alloc = sd.alloc, ev_up = sd.up;
    SB2_TRY(d_pu.alloc((size_t)n_users * f * 8 + 16, st));
    SB2_TRY(d_qi.alloc((size_t)n_items * f * 8 + 16, st));
    if (yj) SB2_TRY(d_yj.alloc((size_t)n_items * f * 8 + 16, st));
    SB2_TRY(d_bu.alloc((size_t)n_users * 8, st));
    SB2_TRY(d_bi.alloc((size_t)n_items * 8, st));
    SB2_CUDA(cudaEventRecord(ev_alloc, st));
    SB2_CUDA(cudaStreamWaitEvent(side, ev_alloc, 0));   // stream-ordered allocations: usable on `side` from here on
    SB2_CUDA(cudaMemcpyAsync(d_pu.p, pu, (size_t)n_users * f * 8, cudaMemcpyHostToDevice, side));
    SB2_CUDA(cudaMemcpyAsync(d_qi.p, qi, (size_t)n_items * f * 8, cudaMemcpyHostToDevice, side));
    if (yj) SB2_CUDA(cudaMemcpyAsync(d_yj.p, yj, (size_t)n_items * f * 8, cudaMemcpyHostToDevice, side));
    SB2_CUDA(cudaEventRecord(ev_up, side));
    sb2_svd_plan* plan = nullptr;
    int rc = svd_plan_create_dev(n_users, n_items, n, d_u.as<int32_t>(), d_i.as<int32_t>(), d_r.as<double>(), prm,
                                 yj != nullptr, yj ? d_up.as<int64_t>() : nullptr, yj ? d_ui.as<int32_t>() : nullptr, 0, 1,
                                 st, &plan);
    cudaError_t we = cudaStreamWaitEvent(st, ev_up, 0);
    if (rc != SB2_OK || we != cudaSuccess) {
        cudaStreamSynchronize(side);   // the buffers are freed on `st` when this function returns
        if (plan) svd_plan_destroy(plan);
        if (rc == SB2_OK) { set_error("svd_fit: cudaStreamWaitEvent failed: %s", cudaGetErrorString(we)); rc = SB2_ERR_CUDA; }
        return rc;
    }
    SB2_TRY(svd_like_run_plan(plan, prm, d_pu.as<double>(), d_qi.as<double>(), yj ? d_yj.as<double>() : nullptr,
                              d_bu.as<double>(), d_bi.as<double>(), st));
    SB2_TRY(download(pu, d_pu.p, (size_t)n_users * f, st));
    SB2_TRY(download(qi, d_qi.p, (size_t)n_items * f, st));
    if (yj) SB2_TRY(download(yj, d_yj.p, (size_t)n_items * f, st));
    SB2_TRY(download(bu, d_bu.p, (size_t)n_users, st));
    SB2_TRY(download(bi, d_bi.p, (size_t)n_items, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_svd_fit(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                const sb2_sgd_params* prm, double* pu, double* qi, double* bu, double* bi) {
    return svd_like_fit_host(n_users, n_items, n, u, i, r, nullptr, nullptr, prm, pu, qi, nullptr, bu, bi);
}

int sb2_svdpp_fit(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                  const int64_t* u_ptr, const int32_t* ui_idx, const sb2_sgd_params* prm, double* pu, double* qi,
                  double* yj, double* bu, double* bi) {
    if (!yj || !u_ptr || !ui_idx) {
        set_error("svdpp_fit: yj, u_ptr and ui_idx are required");
        return SB2_ERR_INVALID;
    }
    return svd_like_fit_host(n_users, n_items, n, u, i, r, u_ptr, ui_idx, prm, pu, qi, yj, bu, bi);
}

int sb2_svd_plan_create(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u_host, const int32_t* i_host,
                        const double* r_host, const sb2_sgd_params* prm, int with_yj, sb2_svd_plan** out) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    DevBuf d_u, d_i, d_r, d_up, d_ui;
    SB2_TRY(upload(d_u, u_host, (size_t)n, st));
    SB2_TRY(upload(d_i, i_host, (size_t)n, st));
    SB2_TRY(upload(d_r, r_host, (size_t)n, st));
    std::vector<int64_t> up;
    if (with_yj) {
        // ur CSR offsets from the grouped COO
        up.assign((size_t)n_users + 1, 0);
        for (int64_t k = 0; k < n; ++k) up[(size_t)u_host[k] + 1]++;
        for (int64_t q = 0; q < n_users; ++q) up[(size_t)q + 1] += up[(size_t)q];
        SB2_TRY(upload(d_up, up.data(), up.size(), st));
    }
    int rc = svd_plan_create_dev(n_users, n_items, n, d_u.as<int32_t>(), d_i.as<int32_t>(), d_r.as<double>(), prm,
                                 with_yj, with_yj ? d_up.as<int64_t>() : nullptr, with_yj ? d_i.as<int32_t>() : nullptr,
                                 0, 1, st, out);
    cudaStreamSynchronize(st);
    return rc;
}

int sb2_svd_plan_reset(sb2_svd_plan* plan, const double* pu_host, const double* qi_host, const double* yj_host) {
    cudaStream_t st = nullptr;
    int64_t nu, ni;
    int f, wy;
    svd_plan_dims(plan, &nu, &ni, &f, &wy);
    DevBuf d_pu, d_qi, d_yj;
    SB2_TRY(upload(d_pu, pu_host, (size_t)nu * f, st));
    SB2_TRY(upload(d_qi, qi_host, (size_t)ni * f, st));
    if (wy) {
        if (!yj_host) {
            set_error("svd_plan_reset: yj required");
            return SB2_ERR_INVALID;
        }
        SB2_TRY(upload(d_yj, yj_host, (size_t)ni * f, st));
    }
    SB2_TRY(svd_plan_reset_dev(plan, d_pu.as<double>(), d_qi.as<double>(), wy ? d_yj.as<double>() : nullptr, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_svd_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, const sb2_sgd_params* prm, int with_yj, const int64_t* u_ptr,
                            const int32_t* ui_idx, void* stream, sb2_svd_plan** out) {
    SB2_TRY(ensure_device());
    return svd_plan_create_dev(n_users, n_items, n, u, i, r, prm, with_yj, u_ptr, ui_idx, 0, 1, (cudaStream_t)stream,
                               out);
}
int sb2_svd_ring_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, const sb2_sgd_params* prm, int with_yj, const int64_t* u_ptr,
                            const int32_t* ui_idx, int rank, int world, void* stream, sb2_svd_plan** out) {
    SB2_TRY(ensure_device());
    return svd_plan_create_dev(n_users, n_items, n, u, i, r, prm, with_yj, u_ptr, ui_idx, rank, world,
                               (cudaStream_t)stream, out);
}
int sb2_svd_ring_ipc_handle(const sb2_svd_plan* plan, unsigned char* handle64) {
    return svd_ring_ipc_handle(plan, handle64);
}
int sb2_svd_ring_connect_ipc(sb2_svd_plan* plan, const unsigned char* left64, const unsigned char* right64) {
    return svd_ring_connect_ipc(plan, left64, right64);
}
int sb2_svd_ring_connect_local(sb2_svd_plan* plan, sb2_svd_plan* left, sb2_svd_plan* right) {
    if (!plan || !left || !right) {
        set_error("svd_ring_connect_local: null plan");
        return SB2_ERR_INVALID;
    }
    return svd_ring_connect_local(plan, left, right);
}
int sb2_svd_ring_run_local(sb2_svd_plan** plans, int n_plans, int n_epochs, void* stream) {
    if (!plans) {
        set_error("svd_ring_run_local: null plans");
        return SB2_ERR_INVALID;
    }
    return svd_ring_run_local(plans, n_plans, n_epochs, (cudaStream_t)stream);
}
int sb2_svd_ring_epoch_local(sb2_svd_plan** plans, int n_plans, float** exchange, void* stream) {
    if (!plans || n_plans < 1 || n_plans > 4) {
        set_error("svd_ring_epoch_local: 1..4 plans");
        return SB2_ERR_INVALID;
    }
    return svd_ring_epoch_local(plans, n_plans, exchange, (cudaStream_t)stream);
}
int sb2_svd_ring_epoch_dev(sb2_svd_plan* plan, int phase, float* exchange, void* stream) {
    return svd_ring_epoch_dev(plan, phase, exchange, (cudaStream_t)stream);
}
int sb2_svd_ring_info(const sb2_svd_plan* plan, int64_t* n_users_local, int64_t* n_items_local, int64_t* n_ratings_local,
                      int* row_stride) {
    svd_ring_info(plan, n_users_local, n_items_local, n_ratings_local, row_stride);
    return SB2_OK;
}
int sb2_svd_plan_status(sb2_svd_plan* plan, void* stream) { return svd_plan_status(plan, (cudaStream_t)stream); }
int sb2_svd_plan_reset_dev(sb2_svd_plan* plan, const double* pu, const double* qi, const double* yj, void* stream) {
    return svd_plan_reset_dev(plan, pu, qi, yj, (cudaStream_t)stream);
}
int sb2_svd_plan_read_dev(sb2_svd_plan* plan, double* pu, double* qi, double* bu, double* bi, double* yj,
                          void* stream) {
    return svd_plan_read_dev(plan, pu, qi, bu, bi, yj, (cudaStream_t)stream);
}

int sb2_svd_plan_run(sb2_svd_plan* plan, int n_epochs, void* stream) {
    return svd_plan_run(plan, n_epochs, (cudaStream_t)stream);
}

int sb2_svd_plan_read(sb2_svd_plan* plan, double* pu, double* qi, double* bu, double* bi, double* yj) {
    cudaStream_t st = nullptr;
    int64_t nu, ni;
    int f, wy;
    svd_plan_dims(plan, &nu, &ni, &f, &wy);
    DevBuf d_pu, d_qi, d_bu, d_bi, d_yj;
    SB2_TRY(d_pu.alloc((size_t)nu * f * 8, st));
    SB2_TRY(d_qi.alloc((size_t)ni * f * 8, st));
    SB2_TRY(d_bu.alloc((size_t)nu * 8, st));
    SB2_TRY(d_bi.alloc((size_t)ni * 8, st));
    if (wy && yj) SB2_TRY(d_yj.alloc((size_t)ni * f * 8, st));
    SB2_TRY(svd_plan_read_dev(plan, d_pu.as<double>(), d_qi.as<double>(), d_bu.as<double>(), d_bi.as<double>(),
                              (wy && yj) ? d_yj.as<double>() : nullptr, st));
    if (pu) SB2_TRY(download(pu, d_pu.p, (size_t)nu * f, st));
    if (qi) SB2_TRY(download(qi, d_qi.p, (size_t)ni * f, st));
    if (bu) SB2_TRY(download(bu, d_bu.p, (size_t)nu, st));
    if (bi) SB2_TRY(download(bi, d_bi.p, (size_t)ni, st));
    if (wy && yj) SB2_TRY(download(yj, d_yj.p, (size_t)ni * f, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

void sb2_svd_plan_destroy(sb2_svd_plan* plan) { svd_plan_destroy(plan); }
int64_t sb2_svd_plan_bytes_per_update(const sb2_svd_plan* plan) { return svd_plan_bytes_per_update(plan); }
int sb2_svd_plan_profile(const sb2_svd_plan* plan, int64_t* cycles_host) {
    return svd_plan_profile(plan, reinterpret_cast<long long*>(cycles_host));
}
int sb2_svd_plan_grid(const sb2_svd_plan* plan, int* n_blocks, int* n_sub) {
    svd_plan_grid(plan, n_blocks, n_sub);
    return SB2_OK;
}
int sb2_svd_plan_layout(const sb2_svd_plan* plan, int* n_blocks, int* cluster, int* lanes, int* chunks, int* n_sub,
                        int* stage_u, int* stage_i, int* dep_mode, int64_t* smem_bytes, int* rec_cap, int* max_cell) {
    if (!plan) {
        set_error("svd_plan_layout: null plan");
        return SB2_ERR_INVALID;
    }
    svd_plan_layout(plan, n_blocks, cluster, lanes, chunks, n_sub, stage_u, stage_i, dep_mode, smem_bytes, rec_cap,
                    max_cell);
    return SB2_OK;
}

// ---- NMF ---------------------------------------------------------------------------------------
int sb2_nmf_fit_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                    const sb2_nmf_params* prm, double* pu, double* qi, double* bu, double* bi, void* stream) {
    SB2_TRY(ensure_device());
    return nmf_fit_dev(n_users, n_items, n, u, i, r, prm, pu, qi, bu, bi, (cudaStream_t)stream);
}

int sb2_nmf_fit(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i, const double* r,
                const sb2_nmf_params* prm, double* pu, double* qi, double* bu, double* bi) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    const size_t f = (size_t)prm->n_factors;
    DevBuf d_u, d_i, d_r, d_pu, d_qi, d_bu, d_bi;
    SB2_TRY(upload(d_u, u, (size_t)n, st));
    SB2_TRY(upload(d_i, i, (size_t)n, st));
    SB2_TRY(upload(d_r, r, (size_t)n, st));
    SB2_TRY(upload(d_pu, pu, (size_t)n_users * f, st));
    SB2_TRY(upload(d_qi, qi, (size_t)n_items * f, st));
    SB2_TRY(d_bu.alloc((size_t)n_users * 8, st));
    SB2_TRY(d_bi.alloc((size_t)n_items * 8, st));
    SB2_TRY(nmf_fit_dev(n_users, n_items, n, d_u.as<int32_t>(), d_i.as<int32_t>(), d_r.as<double>(), prm,
                        d_pu.as<double>(), d_qi.as<double>(), d_bu.as<double>(), d_bi.as<double>(), st));
    SB2_TRY(download(pu, d_pu.p, (size_t)n_users * f, st));
    SB2_TRY(download(qi, d_qi.p, (size_t)n_items * f, st));
    SB2_TRY(download(bu, d_bu.p, (size_t)n_users, st));
    SB2_TRY(download(bi, d_bi.p, (size_t)n_items, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_nmf_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                            const double* r, int n_factors, void* stream, sb2_nmf_plan** out) {
    SB2_TRY(ensure_device());
    return nmf_plan_create_dev(n_users, n_items, n, u, i, r, n_factors, (cudaStream_t)stream, out);
}
int sb2_nmf_plan_epoch_dev(sb2_nmf_plan* plan, const sb2_nmf_params* prm, const double* pu_cur, const double* qi_cur,
                           double* pu_new, double* qi_new, double* bu, double* bi, int64_t user_begin,
                           int64_t user_end, int64_t item_begin, int64_t item_end, void* stream) {
    return nmf_plan_epoch_dev(plan, prm, pu_cur, qi_cur, pu_new, qi_new, bu, bi, user_begin, user_end, item_begin,
                              item_end, (cudaStream_t)stream);
}
int sb2_nmf_plan_status(sb2_nmf_plan* plan, void* stream) { return nmf_plan_status(plan, (cudaStream_t)stream); }
void sb2_nmf_plan_destroy(sb2_nmf_plan* plan) { nmf_plan_destroy(plan); }

// ---- predict -----------------------------------------------------------------------------------
int sb2_mf_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int n_factors, int biased,
                       double global_mean, const double* pu, const double* qi, const double* bu, const double* bi,
                       const double* yj, const int64_t* u_ptr, const int32_t* ui_idx, double* est,
                       uint8_t* impossible, void* stream) {
    SB2_TRY(ensure_device());
    return mf_predict_dev(n_pairs, u, i, n_factors, biased, global_mean, pu, qi, bu, bi, yj, u_ptr, ui_idx, est,
                          impossible, (cudaStream_t)stream);
}

int sb2_mf_predict(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_users, int64_t n_items,
                   int n_factors, int biased, double global_mean, const double* pu, const double* qi, const double* bu,
                   const double* bi, const double* yj, const int64_t* u_ptr, const int32_t* ui_idx, double* est,
                   uint8_t* impossible) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    const size_t f = (size_t)n_factors;
    DevBuf d_u, d_i, d_pu, d_qi, d_bu, d_bi, d_yj, d_up, d_ui, d_est, d_imp;
    SB2_TRY(upload(d_u, u, (size_t)n_pairs, st));
    SB2_TRY(upload(d_i, i, (size_t)n_pairs, st));
    SB2_TRY(upload(d_pu, pu, (size_t)n_users * f, st));
    SB2_TRY(upload(d_qi, qi, (size_t)n_items * f, st));
    SB2_TRY(upload(d_bu, bu, (size_t)n_users, st));
    SB2_TRY(upload(d_bi, bi, (size_t)n_items, st));
    if (yj) {
        SB2_TRY(upload(d_yj, yj, (size_t)n_items * f, st));
        SB2_TRY(upload(d_up, u_ptr, (size_t)n_users + 1, st));
        SB2_TRY(upload(d_ui, ui_idx, (size_t)u_ptr[n_users], st));
    }
    SB2_TRY(d_est.alloc((size_t)std::max<int64_t>(n_pairs, 1) * 8, st));
    SB2_TRY(d_imp.alloc((size_t)std::max<int64_t>(n_pairs, 1), st));
    SB2_TRY(mf_predict_dev(n_pairs, d_u.as<int32_t>(), d_i.as<int32_t>(), n_factors, biased, global_mean,
                           d_pu.as<double>(), d_qi.as<double>(), d_bu.as<double>(), d_bi.as<double>(),
                           yj ? d_yj.as<double>() : nullptr, yj ? d_up.as<int64_t>() : nullptr,
                           yj ? d_ui.as<int32_t>() : nullptr, d_est.as<double>(), d_imp.as<uint8_t>(), st));
    SB2_TRY(download(est, d_est.p, (size_t)n_pairs, st));
    SB2_TRY(download(impossible, d_imp.p, (size_t)n_pairs, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_knn_predict_dev(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, const double* sim,
                        int64_t sim_ld, const int64_t* y_ptr, const int32_t* x_idx, const double* r, int k, int min_k,
                        int mode, double global_mean, const double* bx, const double* by, double* est,
                        int32_t* actual_k, uint8_t* impossible, void* stream) {
    SB2_TRY(ensure_device());
    return knn_predict_dev(n_pairs, x, y, n_x, sim, sim_ld, x, y_ptr, x_idx, r, k, min_k, mode, global_mean, bx, by, est,
                           actual_k, impossible, (cudaStream_t)stream);
}

int sb2_knn_predict_rows_dev(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, const double* sim,
                             int64_t sim_ld, const int32_t* sim_row, const int64_t* y_ptr, const int32_t* x_idx,
                             const double* r, int k, int min_k, int mode, double global_mean, const double* bx,
                             const double* by, double* est, int32_t* actual_k, uint8_t* impossible, void* stream) {
    SB2_TRY(ensure_device());
    if (n_pairs > 0 && !sim_row) {
        set_error("knn_predict_rows: null sim_row");
        return SB2_ERR_INVALID;
    }
    return knn_predict_dev(n_pairs, x, y, n_x, sim, sim_ld, sim_row, y_ptr, x_idx, r, k, min_k, mode, global_mean, bx,
                           by, est, actual_k, impossible, (cudaStream_t)stream);
}

int sb2_knn_predict(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, int64_t n_y, const double* sim,
                    const int64_t* y_ptr, const int32_t* x_idx, const double* r, int k, int min_k, int mode,
                    double global_mean, const double* bx, const double* by, double* est, int32_t* actual_k,
                    uint8_t* impossible) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    const int64_t nnz = y_ptr[n_y];
    DevBuf d_x, d_y, d_sim, d_ptr, d_idx, d_r, d_bx, d_by, d_est, d_ak, d_imp;
    SB2_TRY(upload(d_x, x, (size_t)n_pairs, st));
    SB2_TRY(upload(d_y, y, (size_t)n_pairs, st));
    SB2_TRY(upload(d_sim, sim, (size_t)n_x * (size_t)n_x, st));
    SB2_TRY(upload(d_ptr, y_ptr, (size_t)n_y + 1, st));
    SB2_TRY(upload(d_idx, x_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_r, r, (size_t)nnz, st));
    if (mode != 0) {
        if (!bx || (mode != 3 && !by)) {
            set_error("knn_predict: per-x / per-y vectors required for this mode");
            return SB2_ERR_INVALID;
        }
        SB2_TRY(upload(d_bx, bx, (size_t)n_x, st));
        if (by) SB2_TRY(upload(d_by, by, (size_t)(mode == 4 ? n_x : n_y), st));
    }
    SB2_TRY(d_est.alloc((size_t)std::max<int64_t>(n_pairs, 1) * 8, st));
    SB2_TRY(d_ak.alloc((size_t)std::max<int64_t>(n_pairs, 1) * 4, st));
    SB2_TRY(d_imp.alloc((size_t)std::max<int64_t>(n_pairs, 1), st));
    SB2_TRY(knn_predict_dev(n_pairs, d_x.as<int32_t>(), d_y.as<int32_t>(), n_x, d_sim.as<double>(), n_x,
                            d_x.as<int32_t>(), d_ptr.as<int64_t>(), d_idx.as<int32_t>(), d_r.as<double>(), k, min_k, mode, global_mean,
                            mode ? d_bx.as<double>() : nullptr, (mode && by) ? d_by.as<double>() : nullptr, d_est.as<double>(),
                            d_ak.as<int32_t>(), d_imp.as<uint8_t>(), st));
    SB2_TRY(download(est, d_est.p, (size_t)n_pairs, st));
    SB2_TRY(download(actual_k, d_ak.p, (size_t)n_pairs, st));
    SB2_TRY(download(impossible, d_imp.p, (size_t)n_pairs, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_slope_one_fit_dev(int64_t n_items, int64_t n_users, const int64_t* u_ptr, const int32_t* i_idx, const double* r,
                          int64_t nnz, int64_t* freq_out, double* dev_out, void* stream) {
    SB2_TRY(ensure_device());
    return slope_one_fit_dev(n_items, n_users, u_ptr, i_idx, r, nnz, freq_out, dev_out, (cudaStream_t)stream);
}

int sb2_slope_one_fit(int64_t n_items, int64_t n_users, const int64_t* u_ptr, const int32_t* i_idx, const double* r,
                      int64_t* freq_out, double* dev_out) {
    SB2_TRY(ensure_device());
    cudaStream_t st = nullptr;
    const int64_t nnz = u_ptr[n_users];
    const size_t nn = (size_t)n_items * (size_t)n_items;
    DevBuf d_ptr, d_idx, d_r, d_freq, d_dev;
    SB2_TRY(upload(d_ptr, u_ptr, (size_t)n_users + 1, st));
    SB2_TRY(upload(d_idx, i_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_r, r, (size_t)nnz, st));
    SB2_TRY(d_freq.alloc(nn * 8, st));
    SB2_TRY(d_dev.alloc(nn * 8, st));
    SB2_TRY(slope_one_fit_dev(n_items, n_users, d_ptr.as<int64_t>(), d_idx.as<int32_t>(), d_r.as<double>(), nnz,
                              d_freq.as<int64_t>(), d_dev.as<double>(), st));
    SB2_TRY(download(freq_out, d_freq.p, nn, st));
    SB2_TRY(download(dev_out, d_dev.p, nn, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_slope_one_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_items, const int64_t* freq,
                              const double* dev, const int64_t* u_ptr, const int32_t* i_idx, const double* user_mean,
                              double* est, uint8_t* impossible, void* stream) {
    SB2_TRY(ensure_device());
    return slope_one_predict_dev(n_pairs, u, i, n_items, freq, dev, u_ptr, i_idx, user_mean, est, impossible,
                                 (cudaStream_t)stream);
}

// ---- CoClustering ------------------------------------------------------------------------------
int sb2_coclustering_fit_dev(int64_t n_users, int64_t n_items, int64_t nnz, const int64_t* u_ptr, const int32_t* ui_idx,
                             const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                             const double* user_mean, const double* item_mean, double global_mean, int n_cltr_u,
                             int n_cltr_i, int n_epochs, int32_t* cltr_u, int32_t* cltr_i, double* avg_cltr_u,
                             double* avg_cltr_i, double* avg_cocltr, void* stream) {
    SB2_TRY(ensure_device());
    return coclustering_fit_dev(n_users, n_items, nnz, u_ptr, ui_idx, u_r, i_ptr, iu_idx, i_r, user_mean, item_mean,
                                global_mean, n_cltr_u, n_cltr_i, n_epochs, cltr_u, cltr_i, avg_cltr_u, avg_cltr_i,
                                avg_cocltr, (cudaStream_t)stream);
}

int sb2_coclustering_fit(int64_t n_users, int64_t n_items, const int64_t* u_ptr, const int32_t* ui_idx, const double* u_r,
                         const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r, const double* user_mean,
                         const double* item_mean, double global_mean, int n_cltr_u, int n_cltr_i, int n_epochs,
                         int32_t* cltr_u, int32_t* cltr_i, double* avg_cltr_u, double* avg_cltr_i, double* avg_cocltr) {
    SB2_TRY(ensure_device());
    if (n_cltr_u < 1 || n_cltr_i < 1 || n_users < 0 || n_items < 0) {
        set_error("coclustering: n_cltr_u and n_cltr_i must be >= 1 (got %d, %d)", n_cltr_u, n_cltr_i);
        return SB2_ERR_INVALID;
    }
    cudaStream_t st = nullptr;
    const int64_t nnz = u_ptr[n_users];
    const size_t cells = (size_t)n_cltr_u * (size_t)n_cltr_i;
    DevBuf d_up, d_ui, d_ur, d_ip, d_iu, d_ir, d_um, d_im, d_cu, d_ci, d_au, d_ai, d_ac;
    SB2_TRY(upload(d_up, u_ptr, (size_t)n_users + 1, st));
    SB2_TRY(upload(d_ui, ui_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_ur, u_r, (size_t)nnz, st));
    SB2_TRY(upload(d_ip, i_ptr, (size_t)n_items + 1, st));
    SB2_TRY(upload(d_iu, iu_idx, (size_t)nnz, st));
    SB2_TRY(upload(d_ir, i_r, (size_t)nnz, st));
    SB2_TRY(upload(d_um, user_mean, (size_t)n_users, st));
    SB2_TRY(upload(d_im, item_mean, (size_t)n_items, st));
    SB2_TRY(upload(d_cu, cltr_u, (size_t)n_users, st));
    SB2_TRY(upload(d_ci, cltr_i, (size_t)n_items, st));
    SB2_TRY(d_au.alloc((size_t)n_cltr_u * 8, st));
    SB2_TRY(d_ai.alloc((size_t)n_cltr_i * 8, st));
    SB2_TRY(d_ac.alloc(cells * 8, st));
    SB2_TRY(coclustering_fit_dev(n_users, n_items, nnz, d_up.as<int64_t>(), d_ui.as<int32_t>(), d_ur.as<double>(),
                                 d_ip.as<int64_t>(), d_iu.as<int32_t>(), d_ir.as<double>(), d_um.as<double>(),
                                 d_im.as<double>(), global_mean, n_cltr_u, n_cltr_i, n_epochs, d_cu.as<int32_t>(),
                                 d_ci.as<int32_t>(), d_au.as<double>(), d_ai.as<double>(), d_ac.as<double>(), st));
    SB2_TRY(download(cltr_u, d_cu.p, (size_t)n_users, st));
    SB2_TRY(download(cltr_i, d_ci.p, (size_t)n_items, st));
    SB2_TRY(download(avg_cltr_u, d_au.p, (size_t)n_cltr_u, st));
    SB2_TRY(download(avg_cltr_i, d_ai.p, (size_t)n_cltr_i, st));
    SB2_TRY(download(avg_cocltr, d_ac.p, cells, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    return SB2_OK;
}

int sb2_coclustering_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_users, int64_t n_items,
                                 int n_cltr_i, const int32_t* cltr_u, const int32_t* cltr_i, const double* user_mean,
                                 const double* item_mean, const double* avg_cltr_u, const double* avg_cltr_i,
                                 const double* avg_cocltr, double global_mean, double* est, void* stream) {
    SB2_TRY(ensure_device());
    return coclustering_predict_dev(n_pairs, u, i, n_users, n_items, n_cltr_i, cltr_u, cltr_i, user_mean, item_mean,
                                    avg_cltr_u, avg_cltr_i, avg_cocltr, global_mean, est, (cudaStream_t)stream);
}

int sb2_get_neighbors_dev(int64_t n_x, const double* sim, int64_t sim_ld, int64_t n_rows, const int32_t* rows, int k,
                          int32_t* out, void* stream) {
    SB2_TRY(ensure_device());
    return get_neighbors_dev(n_x, sim, sim_ld, n_rows, rows, k, out, (cudaStream_t)stream);
}

// ---- top-N -------------------------------------------------------------------------------------
int sb2_mf_score_block_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, int f, int biased, double global_mean,
                           const double* pu, const double* qi, const double* bu, const double* bi, const double* yj,
                           const int64_t* u_ptr, const int32_t* ui_idx, double* scores, int64_t ld, void* stream) {
    SB2_TRY(ensure_device());
    return mf_score_block_dev(n_rows, rows, n_items, f, biased, global_mean, pu, qi, bu, bi, yj, u_ptr, ui_idx, scores,
                              ld, (cudaStream_t)stream);
}

int sb2_top_n_select_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                         const uint8_t* impossible, double default_est, double offset, double low, double high,
                         const int64_t* u_ptr, const int32_t* ui_idx, int n, int32_t* items_out, double* est_out,
                         int32_t* count_out, void* stream) {
    SB2_TRY(ensure_device());
    return top_n_select_dev(n_rows, rows, n_items, scores, ld, impossible, default_est, offset, low, high, u_ptr,
                            ui_idx, n, items_out, est_out, count_out, (cudaStream_t)stream);
}

int sb2_fcp_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r, const double* est,
                       int64_t* counts, void* stream) {
    SB2_TRY(ensure_device());
    return fcp_counts_dev(n_seg, n, seg_ptr, r, est, counts, (cudaStream_t)stream);
}

int sb2_precision_at_k_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r,
                                  const double* est, const int64_t* k_eff, double threshold, int64_t* counts,
                                  void* stream) {
    SB2_TRY(ensure_device());
    return precision_at_k_counts_dev(n_seg, n, seg_ptr, r, est, k_eff, threshold, counts, (cudaStream_t)stream);
}

int sb2_top_n_hits_dev(int64_t n_rows, const int32_t* items, int64_t ld, const int32_t* count, int w,
                       const int64_t* rel_ptr, const int32_t* rel_idx, int64_t rel_len, const double* inv,
                       const double* disc, int32_t* hits, double* rr, double* dcg, void* stream) {
    SB2_TRY(ensure_device());
    return top_n_hits_dev(n_rows, items, ld, count, w, rel_ptr, rel_idx, rel_len, inv, disc, hits, rr, dcg,
                          (cudaStream_t)stream);
}

int sb2_top_n_lists_dev(int64_t n_rows, const int32_t* items, int64_t ld, const double* est, const int32_t* count,
                        int w, int has_threshold, double threshold, int64_t n_items, const double* info,
                        const double* sim, int32_t* covered, double* nov, double* ils, uint8_t* seen, void* stream) {
    SB2_TRY(ensure_device());
    return top_n_lists_dev(n_rows, items, ld, est, count, w, has_threshold, threshold, n_items, info, sim, covered,
                           nov, ils, seen, (cudaStream_t)stream);
}

int sb2_top_n_ranks_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                        const uint8_t* impossible, double default_est, double offset, double low, double high,
                        const int64_t* u_ptr, const int32_t* ui_idx, const int64_t* rel_ptr, const int32_t* rel_idx,
                        int64_t rel_len, int32_t* c, int32_t* k, int64_t* s, int32_t* f, void* stream) {
    SB2_TRY(ensure_device());
    return top_n_ranks_dev(n_rows, rows, n_items, scores, ld, impossible, default_est, offset, low, high, u_ptr, ui_idx,
                           rel_ptr, rel_idx, rel_len, c, k, s, f, (cudaStream_t)stream);
}

int sb2_sim_build_upper_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx,
                            const double* r, int64_t nnz, int rating_denom, int min_support, double global_mean,
                            const double* x_biases, const double* y_biases, double shrinkage, int64_t row_begin,
                            int64_t row_end, double* sim_out, void* stream) {
    SB2_TRY(ensure_device());
    return sim_build_upper_dev(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases,
                               y_biases, shrinkage, row_begin, row_end, sim_out, (cudaStream_t)stream);
}

int sb2_sim_build_rows_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx,
                           const double* r, int64_t nnz, int rating_denom, int min_support, double global_mean,
                           const double* x_biases, const double* y_biases, double shrinkage, const int32_t* rows,
                           int64_t n_rows, double* out, int64_t ld, void* stream) {
    SB2_TRY(ensure_device());
    return sim_build_rows_dev(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases,
                              y_biases, shrinkage, rows, n_rows, out, ld, (cudaStream_t)stream);
}

int sb2_rating_denominator_dev(const double* r, int64_t nnz, int* denom_out, void* stream) {
    SB2_TRY(ensure_device());
    if (!denom_out) {
        set_error("rating_denominator: null output");
        return SB2_ERR_INVALID;
    }
    return rating_denominator_dev(r, nnz, denom_out, (cudaStream_t)stream);
}

}  // extern "C"
