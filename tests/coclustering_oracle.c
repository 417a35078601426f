/*
 * TEST INFRASTRUCTURE -- NOT PRODUCT CODE.
 *
 * Plain-C sequential restatement of the reference's CoClustering (prediction_algorithms/co_clustering.pyx:68-237:
 * fit, compute_averages, estimate), used as the parity checker of the CoClustering tests and as the CPU arm of
 * tools/bench_coclustering.py.  Nothing under surprise_b200/ may import, link or call it.
 *
 * It keeps the reference's iteration and operation order and is compiled with gcc -O2 -ffp-contract=off (strict
 * IEEE fp64, no FMA contraction), like the reference's Cython build.  tests/test_coclustering_cpu.py pins it bit for
 * bit against a literal Python transcription of the reference, and against the compiled reference wherever that is
 * built.  Layout: "ur" / "ir" CSR = ptr[n+1], idx[N], r[N] in list order; ur order is also all_ratings() order.
 */
#include <stdint.h>
#include <stdlib.h>

#define ORC_OK 0
#define ORC_NOMEM 2

/* ------------------------------------------------------------------------------------------
 * CoClustering.fit (prediction_algorithms/co_clustering.pyx:68-155) with compute_averages
 * (:157-237).  u_ptr / ui_idx / u_r: trainset.ur flattened (also the all_ratings() order);
 * i_ptr / iu_idx / i_r: trainset.ir flattened.  cltr_u / cltr_i: the rng.randint draw in, the
 * final clusters out.  Ratings go through `cdef int r` (truncation; ORC_OVERFLOW outside the C int
 * range, where the reference raises OverflowError).  avg_cocltr is n_cltr_u x n_cltr_i row-major.
 * ------------------------------------------------------------------------------------------ */
#define ORC_OVERFLOW 3

static int orc_cint(double x, int *out)
{
    if (!(x > -2147483649.0 && x < 2147483648.0)) return ORC_OVERFLOW;
    *out = (int)x;
    return ORC_OK;
}

static int orc_cc_averages(int64_t n_users, const int64_t *u_ptr, const int32_t *ui_idx, const double *u_r,
                           const int64_t *cltr_u, const int64_t *cltr_i, int ncu, int nci, double global_mean,
                           double *avg_u, double *avg_i, double *avg_co)
{
    int64_t *cnt_u = calloc((size_t)ncu, 8), *cnt_i = calloc((size_t)nci, 8),
            *cnt_co = calloc((size_t)ncu * nci, 8);
    double *sum_u = calloc((size_t)ncu, 8), *sum_i = calloc((size_t)nci, 8), *sum_co = calloc((size_t)ncu * nci, 8);
    int rc = (cnt_u && cnt_i && cnt_co && sum_u && sum_i && sum_co) ? ORC_OK : ORC_NOMEM;
    for (int64_t u = 0; rc == ORC_OK && u < n_users; ++u)
        for (int64_t a = u_ptr[u]; a < u_ptr[u + 1]; ++a) {
            int r;
            if ((rc = orc_cint(u_r[a], &r)) != ORC_OK) break;
            const int64_t uc = cltr_u[u], ic = cltr_i[ui_idx[a]];
            cnt_u[uc] += 1; cnt_i[ic] += 1; cnt_co[uc * nci + ic] += 1;
            sum_u[uc] += r; sum_i[ic] += r; sum_co[uc * nci + ic] += r;
        }
    if (rc == ORC_OK) {
        for (int uc = 0; uc < ncu; ++uc) avg_u[uc] = cnt_u[uc] ? sum_u[uc] / cnt_u[uc] : global_mean;
        for (int ic = 0; ic < nci; ++ic) avg_i[ic] = cnt_i[ic] ? sum_i[ic] / cnt_i[ic] : global_mean;
        for (int64_t k = 0; k < (int64_t)ncu * nci; ++k) avg_co[k] = cnt_co[k] ? sum_co[k] / cnt_co[k] : global_mean;
    }
    free(cnt_u); free(cnt_i); free(cnt_co); free(sum_u); free(sum_i); free(sum_co);
    return rc;
}

int orc_coclustering_fit(int64_t n_users, int64_t n_items, const int64_t *u_ptr, const int32_t *ui_idx,
                         const double *u_r, const int64_t *i_ptr, const int32_t *iu_idx, const double *i_r,
                         const double *user_mean, const double *item_mean, double global_mean, int ncu, int nci,
                         int n_epochs, int64_t *cltr_u, int64_t *cltr_i, double *avg_u, double *avg_i,
                         double *avg_co)
{
    double *errors = malloc((size_t)(ncu > nci ? ncu : nci) * sizeof(double));
    if (!errors) return ORC_NOMEM;
    int rc = ORC_OK;
    for (int epoch = 0; rc == ORC_OK && epoch < n_epochs; ++epoch) {
        rc = orc_cc_averages(n_users, u_ptr, ui_idx, u_r, cltr_u, cltr_i, ncu, nci, global_mean, avg_u, avg_i, avg_co);
        for (int64_t u = 0; rc == ORC_OK && u < n_users; ++u) {
            for (int uc = 0; uc < ncu; ++uc) {
                errors[uc] = 0.0;
                for (int64_t a = u_ptr[u]; a < u_ptr[u + 1]; ++a) {
                    const int32_t i = ui_idx[a];
                    int r;
                    if ((rc = orc_cint(u_r[a], &r)) != ORC_OK) break;
                    const int64_t ic = cltr_i[i];
                    const double est = avg_co[uc * nci + ic] + user_mean[u] - avg_u[uc] + item_mean[i] - avg_i[ic];
                    errors[uc] += (r - est) * (r - est);
                }
            }
            int best = 0;
            for (int c = 1; c < ncu; ++c) if (errors[c] < errors[best]) best = c;
            cltr_u[u] = best;
        }
        for (int64_t i = 0; rc == ORC_OK && i < n_items; ++i) {
            for (int ic = 0; ic < nci; ++ic) {
                errors[ic] = 0.0;
                for (int64_t a = i_ptr[i]; a < i_ptr[i + 1]; ++a) {
                    const int32_t u = iu_idx[a];
                    int r;
                    if ((rc = orc_cint(i_r[a], &r)) != ORC_OK) break;
                    const int64_t uc = cltr_u[u];
                    const double est = avg_co[uc * nci + ic] + user_mean[u] - avg_u[uc] + item_mean[i] - avg_i[ic];
                    errors[ic] += (r - est) * (r - est);
                }
            }
            int best = 0;
            for (int c = 1; c < nci; ++c) if (errors[c] < errors[best]) best = c;
            cltr_i[i] = best;
        }
    }
    if (rc == ORC_OK)
        rc = orc_cc_averages(n_users, u_ptr, ui_idx, u_r, cltr_u, cltr_i, ncu, nci, global_mean, avg_u, avg_i, avg_co);
    free(errors);
    return rc;
}

/* CoClustering.estimate: unknown user or item (u < 0 or i < 0) -> global_mean, else the fit's expression. */
int orc_coclustering_estimate(int64_t n_pairs, const int32_t *u, const int32_t *i, int nci, const int64_t *cltr_u,
                              const int64_t *cltr_i, const double *user_mean, const double *item_mean,
                              const double *avg_u, const double *avg_i, const double *avg_co, double global_mean,
                              double *est)
{
    for (int64_t p = 0; p < n_pairs; ++p) {
        if (u[p] < 0 || i[p] < 0) { est[p] = global_mean; continue; }
        const int64_t uc = cltr_u[u[p]], ic = cltr_i[i[p]];
        est[p] = avg_co[uc * nci + ic] + user_mean[u[p]] - avg_u[uc] + item_mean[i[p]] - avg_i[ic];
    }
    return ORC_OK;
}
