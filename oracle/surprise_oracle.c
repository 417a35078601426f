/*
 * TEST INFRASTRUCTURE -- NOT PRODUCT CODE.
 *
 * Plain-C CPU restatement of the fit-time hot path of nickmvincent/Surprise, used only as the
 * parity checker by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs.  Nothing under surprise_b200/ may import, link or call this file.
 *
 * Every function states the reference file:line it follows (paths relative to /root/reference).
 * The restatement keeps the reference's iteration order and operation order, and is compiled with
 * -O2 -ffp-contract=off (the reference's Cython C is built with plain gcc -O2: strict IEEE fp64,
 * no FMA contraction), so results are meant to be BIT-IDENTICAL to the Cython build.
 *
 * Parity pin: tests/test_oracle.py checks this file bit for bit against the golden vectors committed
 * under tests/golden/, which tests/golden/make_golden.py generated from the compiled, unmodified
 * reference (oracle/_ref, built by oracle/build_ref.sh) on the reference's own fixtures.
 *
 * Data layout (flat, mirrors what the reference's dict-of-lists iteration visits):
 *   "yr" CSR : y_ptr[n_y+1], x_idx[N], r[N]   -- for y in yr (insertion order), for (x, r) in yr[y]
 *   all_ratings COO: u[N], i[N], r[N]          -- trainset.all_ratings() order (trainset.py:180-190)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_OK 0
#define ORC_ZERO_DIVISION 1 /* the reference would raise ZeroDivisionError (cdivision=False) */
#define ORC_NOMEM 2

enum { ORC_COSINE = 0, ORC_MSD = 1, ORC_PEARSON = 2, ORC_PEARSON_BASELINE = 3 };

/* ------------------------------------------------------------------------------------------
 * similarities.pyx:28-97 (cosine), :100-166 (msd), :169-258 (pearson), :261-361 (pearson_baseline)
 * One entry point; `kind` selects the accumulators and the finalize rule.
 * ------------------------------------------------------------------------------------------ */
int orc_similarity(int kind, int64_t n_x, int64_t n_y, const int64_t *y_ptr, const int32_t *x_idx,
                   const double *r, int min_support, double global_mean, const double *x_biases,
                   const double *y_biases, double shrinkage, double *sim /* n_x*n_x, out */)
{
    const size_t nn = (size_t)n_x * (size_t)n_x;
    int rc = ORC_OK;
    int64_t *freq = calloc(nn, sizeof(int64_t));
    double *prods = calloc(nn, sizeof(double)); /* msd: sq_diff */
    double *sqi = NULL, *sqj = NULL, *si = NULL, *sj = NULL;
    if (kind != ORC_MSD) {
        sqi = calloc(nn, sizeof(double));
        sqj = calloc(nn, sizeof(double));
    }
    if (kind == ORC_PEARSON) {
        si = calloc(nn, sizeof(double));
        sj = calloc(nn, sizeof(double));
    }
    if (!freq || !prods || (kind != ORC_MSD && (!sqi || !sqj)) || (kind == ORC_PEARSON && (!si || !sj))) {
        rc = ORC_NOMEM;
        goto done;
    }
    memset(sim, 0, nn * sizeof(double));
    int min_sprt = min_support;
    if (kind == ORC_PEARSON_BASELINE && min_sprt < 2) min_sprt = 2; /* similarities.pyx:334 */

    /* accumulation: similarities.pyx:78-84 / :149-153 / :231-238 / :336-345 */
    for (int64_t y = 0; y < n_y; ++y) {
        const int64_t b = y_ptr[y], e = y_ptr[y + 1];
        const double partial_bias = (kind == ORC_PEARSON_BASELINE) ? global_mean + y_biases[y] : 0.0;
        for (int64_t a = b; a < e; ++a) {
            const int64_t xi = x_idx[a];
            const double ri = r[a];
            for (int64_t c = b; c < e; ++c) {
                const int64_t xj = x_idx[c];
                const double rj = r[c];
                const size_t o = (size_t)xi * (size_t)n_x + (size_t)xj;
                switch (kind) {
                case ORC_COSINE:
                    freq[o] += 1;
                    prods[o] += ri * rj;
                    sqi[o] += ri * ri; /* ri**2 -> pow(ri, 2.0) -> gcc folds to ri*ri */
                    sqj[o] += rj * rj;
                    break;
                case ORC_MSD: {
                    const double d = ri - rj;
                    prods[o] += d * d;
                    freq[o] += 1;
                    break;
                }
                case ORC_PEARSON:
                    prods[o] += ri * rj;
                    freq[o] += 1;
                    sqi[o] += ri * ri;
                    sqj[o] += rj * rj;
                    si[o] += ri;
                    sj[o] += rj;
                    break;
                default: { /* pearson_baseline */
                    freq[o] += 1;
                    const double di = ri - (partial_bias + x_biases[xi]);
                    const double dj = rj - (partial_bias + x_biases[xj]);
                    prods[o] += di * dj;
                    sqi[o] += di * di;
                    sqj[o] += dj * dj;
                    break;
                }
                }
            }
        }
    }

    /* finalize: similarities.pyx:86-95 / :155-164 / :240-256 / :347-359 */
    for (int64_t xi = 0; xi < n_x; ++xi) {
        sim[(size_t)xi * n_x + xi] = 1.0;
        for (int64_t xj = xi + 1; xj < n_x; ++xj) {
            const size_t o = (size_t)xi * (size_t)n_x + (size_t)xj;
            double s = 0.0;
            if (freq[o] >= min_sprt) {
                switch (kind) {
                case ORC_COSINE: {
                    const double denum = sqrt(sqi[o] * sqj[o]);
                    s = prods[o] / denum; /* numpy scalar division: inf/nan, no exception */
                    break;
                }
                case ORC_MSD:
                    if (freq[o] == 0) { rc = ORC_ZERO_DIVISION; goto done; } /* :162, cdivision off */
                    s = 1.0 / (prods[o] / (double)freq[o] + 1.0);
                    break;
                case ORC_PEARSON: {
                    const double n = (double)freq[o];
                    const double num = n * prods[o] - si[o] * sj[o];
                    const double denum = sqrt((n * sqi[o] - si[o] * si[o]) * (n * sqj[o] - sj[o] * sj[o]));
                    s = (denum == 0.0) ? 0.0 : num / denum;
                    break;
                }
                default: {
                    s = prods[o] / sqrt(sqi[o] * sqj[o]);
                    const double fm1 = (double)(freq[o] - 1);
                    const double den = fm1 + shrinkage;
                    if (den == 0.0) { rc = ORC_ZERO_DIVISION; goto done; }
                    s *= fm1 / den;
                    break;
                }
                }
            }
            sim[o] = s;
            sim[(size_t)xj * n_x + xi] = s;
        }
    }
done:
    free(freq); free(prods); free(sqi); free(sqj); free(si); free(sj);
    return rc;
}

/* Recompute individual entries sim[xi,xj] from the two sparse rows (for sampled checks at shapes
 * where the dense temporaries do not fit).  Needs the "xr" CSR (rows sorted in y-iteration order:
 * each row lists (y, r) with y ascending = the order in which the reference's outer loop meets
 * them), so the per-entry sums are formed in exactly the reference's order. */
int orc_similarity_pairs(int kind, int64_t n_pairs, const int32_t *pi, const int32_t *pj,
                         const int64_t *x_ptr, const int32_t *y_idx, const double *r, int min_support,
                         double global_mean, const double *x_biases, const double *y_biases,
                         double shrinkage, double *out)
{
    int min_sprt = min_support;
    if (kind == ORC_PEARSON_BASELINE && min_sprt < 2) min_sprt = 2;
    for (int64_t p = 0; p < n_pairs; ++p) {
        const int32_t xi = pi[p], xj = pj[p];
        if (xi == xj) { out[p] = 1.0; continue; }
        const int32_t lo = xi < xj ? xi : xj, hi = xi < xj ? xj : xi; /* value is taken at (lo,hi) */
        int64_t a = x_ptr[lo], ae = x_ptr[lo + 1], c = x_ptr[hi], ce = x_ptr[hi + 1];
        int64_t freq = 0;
        double prods = 0, sqi = 0, sqj = 0, si = 0, sj = 0;
        while (a < ae && c < ce) {
            if (y_idx[a] < y_idx[c]) ++a;
            else if (y_idx[a] > y_idx[c]) ++c;
            else {
                const double ri = r[a], rj = r[c];
                const int32_t y = y_idx[a];
                freq += 1;
                if (kind == ORC_MSD) { const double d = ri - rj; prods += d * d; }
                else if (kind == ORC_PEARSON_BASELINE) {
                    const double pb = global_mean + y_biases[y];
                    const double di = ri - (pb + x_biases[lo]);
                    const double dj = rj - (pb + x_biases[hi]);
                    prods += di * dj; sqi += di * di; sqj += dj * dj;
                } else {
                    prods += ri * rj; sqi += ri * ri; sqj += rj * rj; si += ri; sj += rj;
                }
                ++a; ++c;
            }
        }
        double s = 0.0;
        if (freq >= min_sprt) {
            if (kind == ORC_COSINE) s = prods / sqrt(sqi * sqj);
            else if (kind == ORC_MSD) {
                if (freq == 0) return ORC_ZERO_DIVISION;
                s = 1.0 / (prods / (double)freq + 1.0);
            } else if (kind == ORC_PEARSON) {
                const double n = (double)freq;
                const double num = n * prods - si * sj;
                const double denum = sqrt((n * sqi - si * si) * (n * sqj - sj * sj));
                s = (denum == 0.0) ? 0.0 : num / denum;
            } else {
                s = prods / sqrt(sqi * sqj);
                const double fm1 = (double)(freq - 1);
                s *= fm1 / (fm1 + shrinkage);
            }
        }
        out[p] = s;
    }
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------
 * prediction_algorithms/optimize_baselines.pyx:14-54 (baseline_als)
 * ir CSR: i_ptr[I+1], iu_idx[N], i_r[N] in ir[i] list order; ur CSR likewise.
 * ------------------------------------------------------------------------------------------ */
int orc_baseline_als(int64_t n_users, int64_t n_items, const int64_t *u_ptr, const int32_t *ui_idx,
                     const double *u_r, const int64_t *i_ptr, const int32_t *iu_idx, const double *i_r,
                     double global_mean, int n_epochs, double reg_u, double reg_i, double *bu, double *bi)
{
    memset(bu, 0, (size_t)n_users * sizeof(double));
    memset(bi, 0, (size_t)n_items * sizeof(double));
    for (int ep = 0; ep < n_epochs; ++ep) {
        for (int64_t i = 0; i < n_items; ++i) {
            double dev = 0.0;
            for (int64_t a = i_ptr[i]; a < i_ptr[i + 1]; ++a) dev += i_r[a] - global_mean - bu[iu_idx[a]];
            const double den = reg_i + (double)(i_ptr[i + 1] - i_ptr[i]);
            if (den == 0.0) return ORC_ZERO_DIVISION;
            bi[i] = dev / den;
        }
        for (int64_t u = 0; u < n_users; ++u) {
            double dev = 0.0;
            for (int64_t a = u_ptr[u]; a < u_ptr[u + 1]; ++a) dev += u_r[a] - global_mean - bi[ui_idx[a]];
            const double den = reg_u + (double)(u_ptr[u + 1] - u_ptr[u]);
            if (den == 0.0) return ORC_ZERO_DIVISION;
            bu[u] = dev / den;
        }
    }
    return ORC_OK;
}

/* prediction_algorithms/optimize_baselines.pyx:57-84 (baseline_sgd) */
int orc_baseline_sgd(int64_t n_users, int64_t n_items, int64_t n, const int32_t *u, const int32_t *i,
                     const double *r, double global_mean, int n_epochs, double reg, double lr, double *bu,
                     double *bi)
{
    memset(bu, 0, (size_t)n_users * sizeof(double));
    memset(bi, 0, (size_t)n_items * sizeof(double));
    for (int ep = 0; ep < n_epochs; ++ep)
        for (int64_t k = 0; k < n; ++k) {
            const double err = r[k] - (global_mean + bu[u[k]] + bi[i[k]]);
            bu[u[k]] += lr * (err - reg * bu[u[k]]);
            bi[i[k]] += lr * (err - reg * bi[i[k]]);
        }
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------
 * prediction_algorithms/matrix_factorization.pyx:241-262 (SVD.sgd hot loop).
 * pu/qi arrive holding the rng.normal init (:233-236), bu/bi zero; updated in place.
 * `global_mean` must already be 0 when biased is false (:238-239).
 * ------------------------------------------------------------------------------------------ */
int orc_svd_sgd(int64_t n, int f, const int32_t *u, const int32_t *i, const double *r, int n_epochs,
                int biased, double global_mean, double lr_bu, double lr_bi, double lr_pu, double lr_qi,
                double reg_bu, double reg_bi, double reg_pu, double reg_qi, double *pu, double *qi,
                double *bu, double *bi)
{
    for (int ep = 0; ep < n_epochs; ++ep)
        for (int64_t k = 0; k < n; ++k) {
            double *p = pu + (size_t)u[k] * f, *q = qi + (size_t)i[k] * f;
            double dot = 0.0;
            for (int j = 0; j < f; ++j) dot += q[j] * p[j];
            const double err = r[k] - (global_mean + bu[u[k]] + bi[i[k]] + dot);
            if (biased) {
                bu[u[k]] += lr_bu * (err - reg_bu * bu[u[k]]);
                bi[i[k]] += lr_bi * (err - reg_bi * bi[i[k]]);
            }
            for (int j = 0; j < f; ++j) {
                const double puf = p[j], qif = q[j];
                p[j] += lr_pu * (err * qif - reg_pu * puf);
                q[j] += lr_qi * (err * puf - reg_qi * qif);
            }
        }
    return ORC_OK;
}

/* prediction_algorithms/matrix_factorization.pyx:462-498 (SVDpp.sgd hot loop).
 * u_ptr/ui_idx: the ur CSR (Iu = [j for (j,_) in ur[u]], :469). */
int orc_svdpp_sgd(int64_t n, int f, const int32_t *u, const int32_t *i, const double *r,
                  const int64_t *u_ptr, const int32_t *ui_idx, int n_epochs, double global_mean,
                  double lr_bu, double lr_bi, double lr_pu, double lr_qi, double lr_yj, double reg_bu,
                  double reg_bi, double reg_pu, double reg_qi, double reg_yj, double *pu, double *qi,
                  double *yj, double *bu, double *bi)
{
    double *impl = malloc((size_t)f * sizeof(double));
    if (!impl) return ORC_NOMEM;
    for (int ep = 0; ep < n_epochs; ++ep)
        for (int64_t k = 0; k < n; ++k) {
            const int32_t uu = u[k], ii = i[k];
            const int64_t b = u_ptr[uu], e = u_ptr[uu + 1];
            const double sqrt_iu = sqrt((double)(e - b));
            for (int j = 0; j < f; ++j) impl[j] = 0.0;
            for (int64_t a = b; a < e; ++a) {
                const double *y = yj + (size_t)ui_idx[a] * f;
                for (int j = 0; j < f; ++j) impl[j] += y[j] / sqrt_iu;
            }
            double *p = pu + (size_t)uu * f, *q = qi + (size_t)ii * f;
            double dot = 0.0;
            for (int j = 0; j < f; ++j) dot += q[j] * (p[j] + impl[j]);
            const double err = r[k] - (global_mean + bu[uu] + bi[ii] + dot);
            bu[uu] += lr_bu * (err - reg_bu * bu[uu]);
            bi[ii] += lr_bi * (err - reg_bi * bi[ii]);
            for (int j = 0; j < f; ++j) {
                const double puf = p[j], qif = q[j];
                p[j] += lr_pu * (err * qif - reg_pu * puf);
                q[j] += lr_qi * (err * (puf + impl[j]) - reg_qi * qif);
                for (int64_t a = b; a < e; ++a) {
                    double *y = yj + (size_t)ui_idx[a] * f + j;
                    *y += lr_yj * (err * qif / sqrt_iu - reg_yj * *y);
                }
            }
        }
    free(impl);
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------
 * NOT the reference: the SVD++ relaxation of the stratified SGD kernel (surprise_b200/csrc/sgd.cu,
 * DESIGN.md section 6), restated in fp64 as an element-wise schedule oracle for
 * tests/test_gpu_sgd_schedule.py.  The reference updates every y_j, j in I_u, with each rating of u;
 * the kernel keeps z_u = sum_{j in I_u} y_j / sqrt|I_u| and a gradient accumulator g_u per user and
 * applies the accumulated gradients to y_j once per chunk of strata:
 *
 *   for each epoch, for each chunk c (strata [bounds[c], bounds[c+1])):
 *     z_u = isq_u sum_{j in I_u} y_j;  g_u = 0;  cnt_u = 0           (svdpp_user_refresh_kernel)
 *     for k in order whose stratum lies in the chunk:
 *       err = r - (mu + bu + bi + q.(p + z))
 *       bu += lr_bu (err - reg_bu bu);  bi += lr_bi (err - reg_bi bi)
 *       p' = p + lr_pu (err q - reg_pu p);  q' = q + lr_qi (err (p + z) - reg_qi q)
 *       z' = z + lr_yj (err q - reg_yj z);  g += err isq_u q;  cnt_u += 1      (old p, q, z)
 *     for every item j with c_j = sum_{u in U_j} cnt_u > 0:              (svdpp_item_apply_kernel)
 *       y_j = y_j d^c_j + lr_yj (1 - d^c_j) / (c_j (1 - d)) sum_{u in U_j} g_u,  d = 1 - lr_yj reg_yj
 *       (reg_yj = 0: y_j + lr_yj sum g_u)
 *
 * isq_u = 1/sqrt|I_u| (0 without ratings); I_u from the ur CSR (u_ptr, ui_idx), U_j = the raters of j
 * among all n ratings (u, i), whether or not `order` holds them.  stratum[k] is rating k's stratum,
 * order[0 .. n_order) the sequence in which the ratings are applied (every rating of a chunk in the
 * order they appear there).  `variant` = 0 is the relaxation above; its bits each restate one way a
 * kernel could deviate from it, for the mutation tests (tests/test_sgd_schedule_cpu.py):
 * ------------------------------------------------------------------------------------------ */
enum {
    ORC_PP_Y_FROZEN = 1,      /* the y_j application never runs */
    ORC_PP_NO_DECAY = 2,      /* y_j d^c_j + lr_yj sum g_u: the decay of the c_j updates not integrated */
    ORC_PP_ISQ_INV_N = 4,     /* 1/|I_u| instead of 1/sqrt|I_u| */
    ORC_PP_Z_FROZEN = 8,      /* z_u not advanced by the user's own updates */
    ORC_PP_C_RATERS = 16,     /* c_j = raters of j with cnt_u > 0 instead of their ratings */
    ORC_PP_G_KEPT = 32,       /* g_u not reset between chunks */
};

int orc_svdpp_relaxed_sgd(int64_t n_users, int64_t n_items, int64_t n, int f, const int32_t *u,
                          const int32_t *i, const double *r, const int64_t *u_ptr, const int32_t *ui_idx,
                          const int32_t *stratum, int64_t n_order, const int64_t *order, int n_chunks,
                          const int32_t *bounds, int n_epochs, double global_mean, double lr_bu, double lr_bi,
                          double lr_pu, double lr_qi, double lr_yj, double reg_bu, double reg_bi, double reg_pu,
                          double reg_qi, double reg_yj, int variant, double *pu, double *qi, double *yj,
                          double *bu, double *bi)
{
    const size_t su = (size_t)n_users * f;
    double *z = malloc(su * sizeof(double)), *g = calloc(su, sizeof(double));
    double *isq = malloc((size_t)n_users * sizeof(double)), *cnt = calloc((size_t)n_users, sizeof(double));
    double *acc = malloc((size_t)n_items * f * sizeof(double)), *cj = malloc((size_t)n_items * sizeof(double));
    int64_t *seen = malloc((size_t)n_users * sizeof(int64_t));
    int rc = ORC_OK;
    if (!z || !g || !isq || !cnt || !acc || !cj || !seen) { rc = ORC_NOMEM; goto done; }
    for (int64_t x = 0; x < n_users; ++x) {
        const double len = (double)(u_ptr[x + 1] - u_ptr[x]);
        isq[x] = len > 0 ? ((variant & ORC_PP_ISQ_INV_N) ? 1.0 / len : 1.0 / sqrt(len)) : 0.0;
        seen[x] = -1;
    }
    memset(bu, 0, (size_t)n_users * sizeof(double));
    memset(bi, 0, (size_t)n_items * sizeof(double));
    const double x1 = lr_yj * reg_yj, l1 = log1p(-x1);
    int64_t pass = 0;
    for (int ep = 0; ep < n_epochs; ++ep)
        for (int c = 0; c < n_chunks; ++c, ++pass) {
            const int32_t lo = bounds[c], hi = bounds[c + 1];
            if (lo >= hi) continue;
            for (int64_t x = 0; x < n_users; ++x) cnt[x] = 0.0;
            if (!(variant & ORC_PP_G_KEPT)) memset(g, 0, su * sizeof(double));
            for (int64_t a = 0; a < n_order; ++a) {
                const int64_t k = order[a];
                if (stratum[k] < lo || stratum[k] >= hi) continue;
                const int32_t uu = u[k], ii = i[k];
                double *p = pu + (size_t)uu * f, *q = qi + (size_t)ii * f;
                double *zu = z + (size_t)uu * f, *gu = g + (size_t)uu * f;
                if (seen[uu] != pass) { /* z_u as of the chunk's start: y_j does not change inside a chunk */
                    seen[uu] = pass;
                    for (int j = 0; j < f; ++j) {
                        double s = 0.0;
                        for (int64_t b = u_ptr[uu]; b < u_ptr[uu + 1]; ++b) s += yj[(size_t)ui_idx[b] * f + j];
                        zu[j] = isq[uu] * s;
                    }
                }
                double dot = 0.0;
                for (int j = 0; j < f; ++j) dot += q[j] * (p[j] + zu[j]);
                const double err = r[k] - (global_mean + bu[uu] + bi[ii] + dot);
                bu[uu] += lr_bu * (err - reg_bu * bu[uu]);
                bi[ii] += lr_bi * (err - reg_bi * bi[ii]);
                const double eg = err * isq[uu];
                for (int j = 0; j < f; ++j) {
                    const double puf = p[j], qif = q[j], zuf = zu[j];
                    p[j] = puf + lr_pu * (err * qif - reg_pu * puf);
                    q[j] = qif + lr_qi * (err * (puf + zuf) - reg_qi * qif);
                    if (!(variant & ORC_PP_Z_FROZEN)) zu[j] = zuf + lr_yj * (err * qif - reg_yj * zuf);
                    gu[j] += eg * qif;
                }
                cnt[uu] += 1.0;
            }
            if (variant & ORC_PP_Y_FROZEN) continue;
            /* sum_{u in U_j} g_u and c_j, scattered over all n ratings */
            memset(acc, 0, (size_t)n_items * f * sizeof(double));
            memset(cj, 0, (size_t)n_items * sizeof(double));
            for (int64_t k = 0; k < n; ++k) {
                const int32_t uu = u[k], ii = i[k];
                if (cnt[uu] > 0) cj[ii] += (variant & ORC_PP_C_RATERS) ? 1.0 : cnt[uu];
                else if (!(variant & ORC_PP_G_KEPT)) continue; /* g_u = 0 */
                const double *gu = g + (size_t)uu * f;
                double *aj = acc + (size_t)ii * f;
                for (int j = 0; j < f; ++j) aj[j] += gu[j];
            }
            for (int64_t ii = 0; ii < n_items; ++ii) {
                if (cj[ii] == 0) continue;
                double decay = 1.0, gain = lr_yj;
                if (x1 > 0) {
                    decay = exp(cj[ii] * l1);
                    if (!(variant & ORC_PP_NO_DECAY)) gain = lr_yj * -expm1(cj[ii] * l1) / (cj[ii] * x1);
                }
                double *y = yj + (size_t)ii * f;
                const double *aj = acc + (size_t)ii * f;
                for (int j = 0; j < f; ++j) y[j] = y[j] * decay + gain * aj[j];
            }
        }
done:
    free(z); free(g); free(isq); free(cnt); free(acc); free(cj); free(seen);
    return rc;
}

/* prediction_algorithms/matrix_factorization.pyx:684-730 (NMF.sgd epochs).
 * n_ur[u] = len(ur[u]), n_ir[i] = len(ir[i]).  global_mean already 0 when unbiased (:681-682). */
int orc_nmf_sgd(int64_t n_users, int64_t n_items, int64_t n, int f, const int32_t *u, const int32_t *i,
                const double *r, const int64_t *n_ur, const int64_t *n_ir, int n_epochs, int biased,
                double global_mean, double reg_pu, double reg_qi, double reg_bu, double reg_bi,
                double lr_bu, double lr_bi, double *pu, double *qi, double *bu, double *bi)
{
    const size_t su = (size_t)n_users * f, si = (size_t)n_items * f;
    double *un = malloc(su * sizeof(double)), *ud = malloc(su * sizeof(double));
    double *in = malloc(si * sizeof(double)), *id = malloc(si * sizeof(double));
    int rc = ORC_OK;
    if (!un || !ud || !in || !id) { rc = ORC_NOMEM; goto done; }
    for (int ep = 0; ep < n_epochs; ++ep) {
        memset(un, 0, su * sizeof(double)); memset(ud, 0, su * sizeof(double));
        memset(in, 0, si * sizeof(double)); memset(id, 0, si * sizeof(double));
        for (int64_t k = 0; k < n; ++k) {
            const int32_t uu = u[k], ii = i[k];
            const double *p = pu + (size_t)uu * f, *q = qi + (size_t)ii * f;
            double dot = 0.0;
            for (int j = 0; j < f; ++j) dot += q[j] * p[j];
            const double est = global_mean + bu[uu] + bi[ii] + dot;
            const double err = r[k] - est;
            if (biased) {
                bu[uu] += lr_bu * (err - reg_bu * bu[uu]);
                bi[ii] += lr_bi * (err - reg_bi * bi[ii]);
            }
            for (int j = 0; j < f; ++j) {
                un[(size_t)uu * f + j] += q[j] * r[k];
                ud[(size_t)uu * f + j] += q[j] * est;
                in[(size_t)ii * f + j] += p[j] * r[k];
                id[(size_t)ii * f + j] += p[j] * est;
            }
        }
        for (int64_t uu = 0; uu < n_users; ++uu)
            for (int j = 0; j < f; ++j) {
                const size_t o = (size_t)uu * f + j;
                ud[o] += (double)n_ur[uu] * reg_pu * pu[o];
                if (ud[o] == 0.0) { rc = ORC_ZERO_DIVISION; goto done; }
                pu[o] *= un[o] / ud[o];
            }
        for (int64_t ii = 0; ii < n_items; ++ii)
            for (int j = 0; j < f; ++j) {
                const size_t o = (size_t)ii * f + j;
                id[o] += (double)n_ir[ii] * reg_qi * qi[o];
                if (id[o] == 0.0) { rc = ORC_ZERO_DIVISION; goto done; }
                qi[o] *= in[o] / id[o];
            }
    }
done:
    free(un); free(ud); free(in); free(id);
    return rc;
}

/* ------------------------------------------------------------------------------------------
 * matrix_factorization.pyx:269-299 (SVD.estimate), :737-761 (NMF.estimate), :506-522
 * (SVDpp.estimate; yj != NULL).  u/i < 0 encode "unknown" ('UKN__' ids, algo_base.py:140-146).
 * impossible[k]=1 where the reference raises PredictionImpossible (:291, :759).
 * The reference uses np.dot (BLAS summation order unspecified); this uses index order.
 * ------------------------------------------------------------------------------------------ */
int orc_mf_estimate(int64_t n_pairs, const int32_t *u, const int32_t *i, int f, int biased,
                    double global_mean, const double *pu, const double *qi, const double *bu,
                    const double *bi, const double *yj, const int64_t *u_ptr, const int32_t *ui_idx,
                    double *est, uint8_t *impossible)
{
    for (int64_t k = 0; k < n_pairs; ++k) {
        const int ku = u[k] >= 0, ki = i[k] >= 0;
        impossible[k] = 0;
        double e = 0.0;
        if (biased) {
            e = global_mean;
            if (ku) e += bu[u[k]];
            if (ki) e += bi[i[k]];
        } else if (!(ku && ki)) {
            impossible[k] = 1;
            est[k] = 0.0;
            continue;
        }
        if (ku && ki) {
            const double *p = pu + (size_t)u[k] * f, *q = qi + (size_t)i[k] * f;
            double dot = 0.0;
            if (yj) {
                const int64_t b = u_ptr[u[k]], en = u_ptr[u[k] + 1];
                const double sq = sqrt((double)(en - b));
                for (int j = 0; j < f; ++j) {
                    double s = 0.0; /* sum(self.yj[j] ...) starts from int 0, row order */
                    for (int64_t a = b; a < en; ++a) s += yj[(size_t)ui_idx[a] * f + j];
                    dot += q[j] * (p[j] + s / sq);
                }
            } else {
                for (int j = 0; j < f; ++j) dot += q[j] * p[j];
            }
            e = biased ? e + dot : dot;
        }
        est[k] = e;
    }
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------
 * prediction_algorithms/knns.py:99-123 (KNNBasic.estimate), :274-309 (KNNBaseline.estimate).
 * x[k], y[k]: already switched ids (knns.py:44-52); yr CSR as above; sim n_x*n_x.
 * heapq.nlargest(k, ..., key=sim) == sorted(..., reverse=True)[:k]: descending, ties keep list order.
 * baseline != 0: est = mu + bx[x] + by[y] (+ weighted residual mean), never impossible when both known.
 * Unknown ids (x<0 or y<0): basic -> impossible; baseline -> partial baseline, actual_k = -1
 * (the reference returns a bare float there, knns.py:285-286, so `details` has no actual_k).
 * baseline == 3: KNNWithMeans (knns.py:178-208), bx = means[n_x];  baseline == 4: KNNWithZScore (:372-403),
 * bx = means, by = sigmas (both indexed by x).
 * ------------------------------------------------------------------------------------------ */
typedef struct { double s; double r; int32_t nb; int32_t pos; } orc_nb_t;

static int orc_nb_cmp(const void *a, const void *b)
{
    const orc_nb_t *p = a, *q = b;
    if (p->s > q->s) return -1;
    if (p->s < q->s) return 1;
    return (p->pos > q->pos) - (p->pos < q->pos);
}

int orc_knn_estimate(int64_t n_pairs, const int32_t *x, const int32_t *y, int64_t n_x,
                     const double *sim, const int64_t *y_ptr, const int32_t *x_idx, const double *r,
                     int k, int min_k, int baseline, double global_mean, const double *bx,
                     const double *by, double *est, int32_t *actual_k, uint8_t *impossible)
{
    int64_t cap = 0;
    orc_nb_t *buf = NULL;
    for (int64_t p = 0; p < n_pairs; ++p) {
        const int kx = x[p] >= 0, ky = y[p] >= 0;
        impossible[p] = 0;
        actual_k[p] = -1;
        if (baseline >= 3) {
            if (!(kx && ky)) { impossible[p] = 1; est[p] = 0.0; continue; }
            est[p] = bx[x[p]];
        } else if (baseline) {
            double e = global_mean;
            /* est += bu[u]; est += bi[i] in that order (user first).  The caller passes bx/by
             * already switched, so it must also say which of them is the user side; to stay
             * order-exact we add in (user, item) order via the `baseline` flag: 1 = x is user,
             * 2 = x is item. */
            if (baseline == 1) { if (kx) e += bx[x[p]]; if (ky) e += by[y[p]]; }
            else { if (ky) e += by[y[p]]; if (kx) e += bx[x[p]]; }
            est[p] = e;
            if (!(kx && ky)) continue;
        } else if (!(kx && ky)) {
            impossible[p] = 1;
            est[p] = 0.0;
            continue;
        }
        const int64_t b = y_ptr[y[p]], e2 = y_ptr[y[p] + 1], len = e2 - b;
        if (len > cap) {
            free(buf);
            cap = len * 2;
            buf = malloc((size_t)cap * sizeof(orc_nb_t));
            if (!buf) return ORC_NOMEM;
        }
        for (int64_t a = 0; a < len; ++a) {
            buf[a].nb = x_idx[b + a];
            buf[a].s = sim[(size_t)x[p] * n_x + x_idx[b + a]];
            buf[a].r = r[b + a];
            buf[a].pos = (int32_t)a;
        }
        qsort(buf, (size_t)len, sizeof(orc_nb_t), orc_nb_cmp);
        const int64_t top = len < k ? len : k;
        double sum_sim = 0.0, sum_r = 0.0;
        int ak = 0;
        for (int64_t a = 0; a < top; ++a) {
            if (buf[a].s > 0) {
                sum_sim += buf[a].s;
                if (baseline == 3) {
                    sum_r += buf[a].s * (buf[a].r - bx[buf[a].nb]);
                } else if (baseline == 4) {
                    sum_r += buf[a].s * (buf[a].r - bx[buf[a].nb]) / by[buf[a].nb];
                } else if (baseline) {
                    const double nb_bsl = global_mean + bx[buf[a].nb] + by[y[p]];
                    sum_r += buf[a].s * (buf[a].r - nb_bsl);
                } else {
                    sum_r += buf[a].s * buf[a].r;
                }
                ++ak;
            }
        }
        actual_k[p] = ak;
        if (baseline) {
            if (ak < min_k) sum_r = 0.0;
            if (ak > 0) { /* ZeroDivisionError swallowed otherwise, knns.py:303-306 / :203-206 / :398-401 */
                if (baseline == 4) est[p] += sum_r / sum_sim * by[x[p]];
                else est[p] += sum_r / sum_sim;
            }
        } else {
            if (ak < min_k) { impossible[p] = 1; est[p] = 0.0; continue; }
            if (ak == 0) { impossible[p] = 2; est[p] = 0.0; continue; } /* min_k<=0: 0/0 raises */
            est[p] = sum_r / sum_sim;
        }
    }
    free(buf);
    return ORC_OK;
}

/* ------------------------------------------------------------------------------------------
 * SlopeOne.fit (prediction_algorithms/slope_one.pyx:44-80).  u_ptr / i_idx / r: trainset.ur flattened.
 * `cdef int ... r_ui, r_uj` (:52): the ratings are converted to C ints (truncation) before the
 * subtraction; dev accumulates the int difference as a double, is divided by freq for i < j
 * (0 / 0 -> NaN, no exception: the module is compiled with cdivision semantics for this statement)
 * and mirrored with a sign flip; dev[i][i] = 0.  freq is int64 and keeps its diagonal.
 * ------------------------------------------------------------------------------------------ */
int orc_slope_one_fit(int64_t n_items, int64_t n_users, const int64_t *u_ptr, const int32_t *i_idx,
                      const double *r, int64_t *freq, double *dev)
{
    const size_t nn = (size_t)n_items * (size_t)n_items;
    memset(freq, 0, nn * sizeof(int64_t));
    for (size_t k = 0; k < nn; ++k) dev[k] = 0.0;
    for (int64_t u = 0; u < n_users; ++u)
        for (int64_t a = u_ptr[u]; a < u_ptr[u + 1]; ++a) {
            const int r_ui = (int)r[a];
            for (int64_t b = u_ptr[u]; b < u_ptr[u + 1]; ++b) {
                const int r_uj = (int)r[b];
                const size_t o = (size_t)i_idx[a] * (size_t)n_items + (size_t)i_idx[b];
                freq[o] += 1;
                dev[o] += r_ui - r_uj;
            }
        }
    for (int64_t i = 0; i < n_items; ++i) {
        dev[(size_t)i * n_items + i] = 0;
        for (int64_t j = i + 1; j < n_items; ++j) {
            const size_t o = (size_t)i * n_items + j;
            dev[o] /= (double)freq[o];
            dev[(size_t)j * n_items + i] = -dev[o];
        }
    }
    return ORC_OK;
}

/* SlopeOne.estimate (slope_one.pyx:82-97): Ri = items j of ur[u] with freq[i, j] > 0;
 * est = user_mean[u] + sum(dev[i, j] for j in Ri) / len(Ri), sum() left to right from 0. */
int orc_slope_one_estimate(int64_t n_pairs, const int32_t *u, const int32_t *i, int64_t n_items,
                           const int64_t *freq, const double *dev, const int64_t *u_ptr,
                           const int32_t *i_idx, const double *user_mean, double *est,
                           uint8_t *impossible)
{
    for (int64_t p = 0; p < n_pairs; ++p) {
        impossible[p] = 0;
        if (u[p] < 0 || i[p] < 0) { impossible[p] = 1; est[p] = 0.0; continue; }
        double sum = 0.0;
        int64_t cnt = 0;
        for (int64_t a = u_ptr[u[p]]; a < u_ptr[u[p] + 1]; ++a) {
            const size_t o = (size_t)i[p] * (size_t)n_items + (size_t)i_idx[a];
            if (freq[o] > 0) { sum += dev[o]; ++cnt; }
        }
        double e = user_mean[u[p]];
        if (cnt) e += sum / (double)cnt;
        est[p] = e;
    }
    return ORC_OK;
}
