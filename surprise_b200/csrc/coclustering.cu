// CoClustering (prediction_algorithms/co_clustering.pyx:68-237 fit / compute_averages, then estimate).
//
// Bit-exactness discipline (DESIGN.md §3.5):
//   - ratings are read into C ints (truncation toward zero), as the reference's `cdef int r` does;
//   - compute_averages adds integers into doubles whose partial sums stay exact below 2^53, so an int64
//     histogram of the n_cltr_u x n_cltr_i co-cluster table in any order gives the reference's bits; the
//     per-cluster marginals are its row / column totals;
//   - every errors[c] of the two assignment passes is an ordered fp64 chain in ur[u] (ir[i]) order of
//     (r - est)^2 terms with est = ((((A + um) - acu) + im) - aci), all __d*_rn (no FMA contraction).
//     The terms of a 32-entry chunk are computed by the 32 lanes of a warp in parallel (one entry per lane,
//     every candidate cluster) and parked in shared memory; lane c then adds the column of candidate c
//     into its chain in entry order.  Only that add is serial.
//   - np.argmin: the first minimum (ties go to the lower cluster index).
// The whole fit is enqueued without a host synchronisation; a device status word makes every kernel after an
// invalid input a no-op and is read once at the end.
#include <math_constants.h>

#include <algorithm>
#include <climits>

#include "common.cuh"

namespace sb2 {

enum { CC_BAD_RATING = 1, CC_BAD_CLUSTER = 2 };

constexpr int CC_WARPS = 4;                 // warps (= segments) per CTA of the assignment kernel
constexpr int CC_PAD = 33;                  // row stride (doubles) of the per-warp term tile
constexpr int CC_HIST_THREADS = 256;
constexpr int CC_SMEM_HIST_BYTES = 48 * 1024;

// Ratings -> C ints (both CSRs), range check of ratings and of the initial clusters, and the owner (user) of every
// entry of the ur CSR for the histogram.
__global__ void cc_prepare_kernel(int64_t nnz, int64_t n_users, int64_t n_items, const int64_t* __restrict__ u_ptr,
                                  const double* __restrict__ u_r, const double* __restrict__ i_r,
                                  int32_t* __restrict__ ru, int32_t* __restrict__ ri, int32_t* __restrict__ own_u,
                                  const int32_t* __restrict__ cltr_u, const int32_t* __restrict__ cltr_i, int n_cu,
                                  int n_ci, int* status) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int bad = 0;
    for (int64_t a = t0; a < nnz; a += stride) {
        const double x = u_r[a], y = i_r[a];
        // Cython's `cdef int r = <python float>` raises OverflowError outside the C int range (and on NaN)
        const bool okx = x > -2147483649.0 && x < 2147483648.0, oky = y > -2147483649.0 && y < 2147483648.0;
        if (!(okx && oky)) bad |= CC_BAD_RATING;
        ru[a] = okx ? (int32_t)x : 0;
        ri[a] = oky ? (int32_t)y : 0;
    }
    for (int64_t u = t0; u < n_users; u += stride) {
        if (cltr_u[u] < 0 || cltr_u[u] >= n_cu) bad |= CC_BAD_CLUSTER;
        for (int64_t a = u_ptr[u]; a < u_ptr[u + 1]; ++a) own_u[a] = (int32_t)u;
    }
    for (int64_t i = t0; i < n_items; i += stride)
        if (cltr_i[i] < 0 || cltr_i[i] >= n_ci) bad |= CC_BAD_CLUSTER;
    if (bad) atomicOr(status, bad);
}

// compute_averages, part 1 (co_clustering.pyx:157-237): hist[2 * (uc * n_ci + ic) + {0, 1}] += {1, r} over all
// ratings.  Equal keys of a warp are combined first (__match_any_sync + __reduce_add_sync on 16-bit halves of r,
// which cannot overflow), so one atomic per distinct cell and warp step; the cells live in shared memory when the
// table fits (flushed once per CTA), in global memory otherwise.
__global__ void __launch_bounds__(CC_HIST_THREADS) cc_hist_kernel(
    int64_t nnz, const int32_t* __restrict__ own_u, const int32_t* __restrict__ ui_idx, const int32_t* __restrict__ ru,
    const int32_t* __restrict__ cltr_u, const int32_t* __restrict__ cltr_i, int n_ci, int cells, int use_smem,
    unsigned long long* __restrict__ hist, const int* status) {
    extern __shared__ unsigned long long cc_sh_hist[];
    if (*status) return;
    unsigned long long* h = use_smem ? cc_sh_hist : hist;
    if (use_smem) {
        for (int k = threadIdx.x; k < 2 * cells; k += blockDim.x) cc_sh_hist[k] = 0ull;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = blockIdx.x * (int64_t)blockDim.x; base < nnz; base += stride) {  // uniform per CTA
        const int64_t a = base + threadIdx.x;
        const bool act = a < nnz;
        int key = -1, r = 0;
        if (act) {
            key = cltr_u[own_u[a]] * n_ci + cltr_i[ui_idx[a]];
            r = ru[a];
        }
        const unsigned m = __match_any_sync(0xffffffffu, key);
        const unsigned lo = __reduce_add_sync(m, (unsigned)(r & 0xffff));
        const int hi = __reduce_add_sync(m, r >> 16);
        if (act && lane == __ffs(m) - 1) {
            atomicAdd(&h[2 * (int64_t)key], (unsigned long long)__popc(m));
            atomicAdd(&h[2 * (int64_t)key + 1], (unsigned long long)((long long)hi * 65536 + (long long)lo));
        }
    }
    if (use_smem) {
        __syncthreads();
        for (int k = threadIdx.x; k < 2 * cells; k += blockDim.x)
            if (cc_sh_hist[k]) atomicAdd(&hist[k], cc_sh_hist[k]);
    }
}

// compute_averages, part 2 (co_clustering.pyx:157-237): marginals and the three average arrays, global_mean for an
// empty cluster.  Clears the histogram for the next call.  One CTA.
__global__ void cc_finalize_kernel(int n_cu, int n_ci, unsigned long long* hist, double mu, double* avg_u,
                                   double* avg_i, double* avg_co, const int* status) {
    if (*status) return;
    const long long* hs = reinterpret_cast<const long long*>(hist);
    for (int uc = threadIdx.x; uc < n_cu; uc += blockDim.x) {
        long long c = 0, s = 0;
        for (int ic = 0; ic < n_ci; ++ic) {
            c += hs[2 * ((int64_t)uc * n_ci + ic)];
            s += hs[2 * ((int64_t)uc * n_ci + ic) + 1];
        }
        avg_u[uc] = c ? __ddiv_rn((double)s, (double)c) : mu;
    }
    for (int ic = threadIdx.x; ic < n_ci; ic += blockDim.x) {
        long long c = 0, s = 0;
        for (int uc = 0; uc < n_cu; ++uc) {
            c += hs[2 * ((int64_t)uc * n_ci + ic)];
            s += hs[2 * ((int64_t)uc * n_ci + ic) + 1];
        }
        avg_i[ic] = c ? __ddiv_rn((double)s, (double)c) : mu;
    }
    __syncthreads();
    const int64_t cells = (int64_t)n_cu * n_ci;
    for (int64_t k = threadIdx.x; k < cells; k += blockDim.x) {
        const long long c = hs[2 * k], s = hs[2 * k + 1];
        avg_co[k] = c ? __ddiv_rn((double)s, (double)c) : mu;
        hist[2 * k] = hist[2 * k + 1] = 0ull;
    }
}

// One assignment pass of CoClustering.fit's epoch loop (co_clustering.pyx:68-155; users first, then items): a warp per segment s.
//   ITEM == false: s = user u, candidates uc, entries (i, r) of ur[u], oc = cltr_i[i] (previous epoch);
//   ITEM == true:  s = item i, candidates ic, entries (u, r) of ir[i], oc = cltr_u[u] (this epoch's, new).
// est = ((((avg_co[uc, ic] + user_mean[u]) - avg_u[uc]) + item_mean[i]) - avg_i[ic]) on both sides.
template <bool ITEM>
__global__ void __launch_bounds__(CC_WARPS * 32) cc_assign_kernel(
    int64_t n_seg, const int64_t* __restrict__ ptr, const int32_t* __restrict__ oidx, const int32_t* __restrict__ rint,
    int32_t* __restrict__ mine_cltr, const int32_t* __restrict__ other_cltr, const double* __restrict__ mean_seg,
    const double* __restrict__ mean_other, const double* __restrict__ avg_co, const double* __restrict__ avg_u,
    const double* __restrict__ avg_i, int n_mine, int n_other, const int* status) {
    extern __shared__ double cc_tile[];
    if (*status) return;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t s = blockIdx.x * (int64_t)CC_WARPS + w;
    if (s >= n_seg) return;  // whole warps leave together
    const int rows = min(32, n_mine);
    double* tile = cc_tile + (size_t)w * rows * CC_PAD;
    const int64_t b = ptr[s], e = ptr[s + 1];
    const double ms = mean_seg[s];
    const double* avg_mine = ITEM ? avg_i : avg_u;
    const double* avg_oth = ITEM ? avg_u : avg_i;
    const int n_ci = ITEM ? n_mine : n_other;
    double best = CUDART_INF;
    int best_c = 0;
    for (int c0 = 0; c0 < n_mine; c0 += 32) {
        const int nc = min(32, n_mine - c0);
        double err = 0.0;
        for (int64_t base = b; base < e; base += 32) {
            const int cnt = e - base < 32 ? (int)(e - base) : 32;
            if (lane < cnt) {
                const int64_t a = base + lane;
                const int32_t o = oidx[a];
                const double r = (double)rint[a];
                const int oc = other_cltr[o];
                const double mo = mean_other[o];
                const double ao = avg_oth[oc];
                for (int j = 0; j < nc; ++j) {
                    const int c = c0 + j;
                    double est;
                    if (!ITEM) {
                        est = __dadd_rn(avg_co[(int64_t)c * n_ci + oc], ms);
                        est = __dsub_rn(est, avg_mine[c]);
                        est = __dadd_rn(est, mo);
                        est = __dsub_rn(est, ao);
                    } else {
                        est = __dadd_rn(avg_co[(int64_t)oc * n_ci + c], mo);
                        est = __dsub_rn(est, ao);
                        est = __dadd_rn(est, ms);
                        est = __dsub_rn(est, avg_mine[c]);
                    }
                    const double d = __dsub_rn(r, est);
                    tile[j * CC_PAD + lane] = __dmul_rn(d, d);
                }
            }
            __syncwarp();
            if (lane < nc) {
                const double* row = tile + lane * CC_PAD;
                for (int k = 0; k < cnt; ++k) err = __dadd_rn(err, row[k]);
            }
            __syncwarp();
        }
        // first minimum of this group of candidates, then against the earlier (lower-index) groups
        double v = lane < nc ? err : CUDART_INF;
        int ci = lane < nc ? c0 + lane : INT_MAX;
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, v, off);
            const int oi = __shfl_xor_sync(0xffffffffu, ci, off);
            if (ov < v || (ov == v && oi < ci)) {
                v = ov;
                ci = oi;
            }
        }
        if (v < best) {
            best = v;
            best_c = ci;
        }
    }
    if (lane == 0) mine_cltr[s] = best_c;
}

// CoClustering.estimate: one thread per pair; unknown user or item -> global_mean (not PredictionImpossible).
__global__ void cc_predict_kernel(int64_t n, const int32_t* __restrict__ u, const int32_t* __restrict__ i,
                                  int64_t n_users, int64_t n_items, int n_ci, const int32_t* __restrict__ cltr_u,
                                  const int32_t* __restrict__ cltr_i, const double* __restrict__ user_mean,
                                  const double* __restrict__ item_mean, const double* __restrict__ avg_u,
                                  const double* __restrict__ avg_i, const double* __restrict__ avg_co, double mu,
                                  double* __restrict__ est) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int32_t uu = u[k], ii = i[k];
    if (uu < 0 || ii < 0 || uu >= n_users || ii >= n_items) {
        est[k] = mu;
        return;
    }
    const int uc = cltr_u[uu], ic = cltr_i[ii];
    double e = __dadd_rn(avg_co[(int64_t)uc * n_ci + ic], user_mean[uu]);
    e = __dsub_rn(e, avg_u[uc]);
    e = __dadd_rn(e, item_mean[ii]);
    est[k] = __dsub_rn(e, avg_i[ic]);
}

int coclustering_fit_dev(int64_t n_users, int64_t n_items, int64_t nnz, const int64_t* u_ptr, const int32_t* ui_idx,
                         const double* u_r, const int64_t* i_ptr, const int32_t* iu_idx, const double* i_r,
                         const double* user_mean, const double* item_mean, double mu, int n_cu, int n_ci, int n_epochs,
                         int32_t* cltr_u, int32_t* cltr_i, double* avg_u, double* avg_i, double* avg_co,
                         cudaStream_t st) {
    if (n_cu < 1 || n_ci < 1) {
        set_error("coclustering: n_cltr_u and n_cltr_i must be >= 1 (got %d, %d)", n_cu, n_ci);
        return SB2_ERR_INVALID;
    }
    const int64_t cells = (int64_t)n_cu * n_ci;
    if (cells > INT32_MAX / 2 || n_users < 0 || n_items < 0 || nnz < 0 || n_users > INT32_MAX || n_items > INT32_MAX) {
        set_error("coclustering: invalid sizes");
        return SB2_ERR_INVALID;
    }
    DevBuf d_ru, d_ri, d_own, d_hist, d_status;
    SB2_TRY(d_ru.alloc((size_t)nnz * 4 + 16, st));
    SB2_TRY(d_ri.alloc((size_t)nnz * 4 + 16, st));
    SB2_TRY(d_own.alloc((size_t)nnz * 4 + 16, st));
    SB2_TRY(d_hist.alloc((size_t)cells * 16, st));
    SB2_TRY(d_status.alloc(sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(d_status.p, 0, sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(d_hist.p, 0, (size_t)cells * 16, st));
    int* status = d_status.as<int>();
    unsigned long long* hist = d_hist.as<unsigned long long>();
    const int sms = sm_count();
    {
        const int64_t work = std::max<int64_t>(std::max(nnz, n_users), std::max<int64_t>(n_items, 1));
        const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(work, 256), (int64_t)sms * 8);
        cc_prepare_kernel<<<grid, 256, 0, st>>>(nnz, n_users, n_items, u_ptr, u_r, i_r, d_ru.as<int32_t>(),
                                                d_ri.as<int32_t>(), d_own.as<int32_t>(), cltr_u, cltr_i, n_cu, n_ci,
                                                status);
        SB2_LAUNCH_CHECK();
    }
    const int use_smem = cells * 16 <= CC_SMEM_HIST_BYTES;
    const unsigned hist_grid =
        (unsigned)std::max<int64_t>(1, std::min<int64_t>(ceil_div(nnz, CC_HIST_THREADS), (int64_t)sms * 4));
    const size_t hist_smem = use_smem ? (size_t)cells * 16 : 0;
    auto averages = [&]() -> int {
        if (nnz > 0) {
            cc_hist_kernel<<<hist_grid, CC_HIST_THREADS, hist_smem, st>>>(nnz, d_own.as<int32_t>(), ui_idx,
                                                                          d_ru.as<int32_t>(), cltr_u, cltr_i, n_ci,
                                                                          (int)cells, use_smem, hist, status);
            SB2_LAUNCH_CHECK();
        }
        cc_finalize_kernel<<<1, 1024, 0, st>>>(n_cu, n_ci, hist, mu, avg_u, avg_i, avg_co, status);
        SB2_LAUNCH_CHECK();
        return SB2_OK;
    };
    const size_t smem_u = (size_t)CC_WARPS * std::min(32, n_cu) * CC_PAD * sizeof(double);
    const size_t smem_i = (size_t)CC_WARPS * std::min(32, n_ci) * CC_PAD * sizeof(double);
    for (int ep = 0; ep < n_epochs; ++ep) {
        SB2_TRY(averages());
        if (n_users > 0) {
            cc_assign_kernel<false><<<(unsigned)ceil_div(n_users, CC_WARPS), CC_WARPS * 32, smem_u, st>>>(
                n_users, u_ptr, ui_idx, d_ru.as<int32_t>(), cltr_u, cltr_i, user_mean, item_mean, avg_co, avg_u,
                avg_i, n_cu, n_ci, status);
            SB2_LAUNCH_CHECK();
        }
        if (n_items > 0) {
            cc_assign_kernel<true><<<(unsigned)ceil_div(n_items, CC_WARPS), CC_WARPS * 32, smem_i, st>>>(
                n_items, i_ptr, iu_idx, d_ri.as<int32_t>(), cltr_i, cltr_u, item_mean, user_mean, avg_co, avg_u,
                avg_i, n_ci, n_cu, status);
            SB2_LAUNCH_CHECK();
        }
    }
    SB2_TRY(averages());
    int h = 0;
    SB2_CUDA(cudaMemcpyAsync(&h, status, sizeof(int), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (h & CC_BAD_RATING) {
        set_error("coclustering: a rating does not fit a C int (the reference raises OverflowError)");
        return SB2_ERR_INVALID;
    }
    if (h & CC_BAD_CLUSTER) {
        set_error("coclustering: an initial cluster index is outside [0, n_cltr)");
        return SB2_ERR_INVALID;
    }
    return SB2_OK;
}

int coclustering_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_users, int64_t n_items,
                             int n_ci, const int32_t* cltr_u, const int32_t* cltr_i, const double* user_mean,
                             const double* item_mean, const double* avg_u, const double* avg_i, const double* avg_co,
                             double mu, double* est, cudaStream_t st) {
    if (n_pairs <= 0) return SB2_OK;
    cc_predict_kernel<<<(unsigned)ceil_div(n_pairs, 256), 256, 0, st>>>(n_pairs, u, i, n_users, n_items, n_ci, cltr_u,
                                                                         cltr_i, user_mean, item_mean, avg_u, avg_i,
                                                                         avg_co, mu, est);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

}  // namespace sb2
