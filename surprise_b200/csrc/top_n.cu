// Top-N recommendations (the reference FAQ's get_top_n over algo.test(trainset.build_anti_testset())):
//   - a dense scorer for the factor models that writes, for a block of users x all items, exactly the bits
//     mf_predict_kernel (predict.cu) returns for each pair;
//   - a per-row selection shared by every algorithm: default_prediction for impossible pairs, offset, clipping,
//     the user's trainset items masked out, and the first n in (score desc, item asc) order -- the order Python's
//     stable sort(reverse=True) leaves the anti-testset (ascending inner item id per user) in.
#include "top_n.cuh"

namespace sb2 {

// ------------------------------------------------------------------------------------------------
// Factor scorer.
// mf_predict_kernel gives lane l the chain part_l = fma(q[j], p[j], part_l), j = l, l + 32, ..., from 0.0, and
// combines the 32 partials with the xor butterfly o = 16, 8, 4, 2, 1.  fp add is commutative, so every lane ends
// with the same value: a fixed binary tree whose level k pairs lanes differing in bit 4 - k.  Visiting the lanes
// in bit-reversed order (l = rev5(k)) makes siblings arrive next to each other, and a 5-deep stack evaluates that
// exact tree per pair (merge while the low bits of k are ones, like a binary counter).
// The factors are repacked slot-major, [l][t] = row[l + 32 t], padded with +0.0 to T = ceil(f / 32) terms per
// slot: a chain starts at +0.0 and can never become -0.0 (x + (+0.0) with x != -0.0 is x; -0 + +0 is +0), so
// fma(+0, +0, c) == c and the padding leaves every partial, and every zero-factor slot, with the same bits.
// SVD++: z[u][j] = p[j] + s / sqrt(|ur[u]|), s summed in ur[u] order from 0.0 -- the expression
// mf_predict_kernel evaluates before its fma -- is computed once per user and scored in place of p.
// Biased: (mu + bu[u]) is hoisted per user; est = ((mu + bu[u]) + bi[i]) + part, as in mf_predict_kernel.
// ------------------------------------------------------------------------------------------------
constexpr int SC_WARPS = 4;
constexpr int SC_RU = 4;                         // rows (users) per thread; a warp shares them (broadcast loads)
constexpr int SC_RI = 2;                         // items per thread: lane and lane + 32
constexpr int SC_ROWS = SC_WARPS * SC_RU;        // rows per block
constexpr int SC_ITEMS = 32 * SC_RI;             // items per block

__global__ void top_n_repack_items_kernel(int64_t n_items, int f, int T, const double* __restrict__ qi,
                                          double* __restrict__ qr) {
    const int64_t total = (int64_t)n_items * 32 * T;
    for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = x % n_items, lt = x / n_items;      // lt = l * T + t
        const int l = (int)(lt / T), t = (int)(lt % T), j = l + 32 * t;
        qr[x] = j < f ? qi[(size_t)i * f + j] : 0.0;
    }
}

__global__ void top_n_repack_users_kernel(int64_t n_rows, const int32_t* __restrict__ rows, int f, int T, int biased,
                                          double mu, const double* __restrict__ pu, const double* __restrict__ bu,
                                          const double* __restrict__ yj, const int64_t* __restrict__ u_ptr,
                                          const int32_t* __restrict__ ui_idx, double* __restrict__ pr,
                                          double* __restrict__ hb) {
    const int64_t total = n_rows * 32 * T;
    for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = x % n_rows, lt = x / n_rows;
        const int l = (int)(lt / T), t = (int)(lt % T), j = l + 32 * t;
        const int32_t uu = rows[r];
        double v = 0.0;
        if (j < f) {
            v = pu[(size_t)uu * f + j];
            if (yj) {
                const int64_t b = u_ptr[uu], en = u_ptr[uu + 1];
                const double sq = sqrt((double)(en - b));
                double s = 0.0;
                for (int64_t a = b; a < en; ++a) s += yj[(size_t)ui_idx[a] * f + j];
                v = v + s / sq;
            }
        }
        pr[x] = v;
        if (lt == 0 && biased) hb[r] = __dadd_rn(mu, bu[uu]);
    }
    if (T == 0 && biased)
        for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n_rows; r += (int64_t)gridDim.x * blockDim.x)
            hb[r] = __dadd_rn(mu, bu[rows[r]]);
}

__global__ void __launch_bounds__(SC_WARPS * 32, 3)
top_n_score_kernel(int64_t n_rows, int64_t n_items, int T, int biased, const double* __restrict__ pr,
                   const double* __restrict__ qr, const double* __restrict__ hb, const double* __restrict__ bi,
                   double* __restrict__ scores, int64_t ld) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t r0 = blockIdx.y * (int64_t)SC_ROWS + w * SC_RU;
    const int64_t i0 = blockIdx.x * (int64_t)SC_ITEMS + lane;
    int64_t rr[SC_RU], ii[SC_RI];
#pragma unroll
    for (int a = 0; a < SC_RU; ++a) rr[a] = r0 + a < n_rows ? r0 + a : n_rows - 1;   // clamped: loads stay in range
#pragma unroll
    for (int b = 0; b < SC_RI; ++b) ii[b] = i0 + 32 * b < n_items ? i0 + 32 * b : n_items - 1;
    double st[5][SC_RU][SC_RI];
#pragma unroll
    for (int k = 0; k < 32; ++k) {
        const int l = (int)(__brev((unsigned)k) >> 27);    // rev5(k)
        double c[SC_RU][SC_RI];
#pragma unroll
        for (int a = 0; a < SC_RU; ++a)
#pragma unroll
            for (int b = 0; b < SC_RI; ++b) c[a][b] = 0.0;
        const double* pl = pr + (size_t)l * T * n_rows;
        const double* ql = qr + (size_t)l * T * n_items;
        for (int t = 0; t < T; ++t) {
            double p[SC_RU], q[SC_RI];
#pragma unroll
            for (int a = 0; a < SC_RU; ++a) p[a] = pl[(size_t)t * n_rows + rr[a]];
#pragma unroll
            for (int b = 0; b < SC_RI; ++b) q[b] = ql[(size_t)t * n_items + ii[b]];
#pragma unroll
            for (int a = 0; a < SC_RU; ++a)
#pragma unroll
                for (int b = 0; b < SC_RI; ++b) c[a][b] = __fma_rn(q[b], p[a], c[a][b]);
        }
        // push leaf k: merge with the stored sibling at every level whose bit of k is set (the trailing ones of k),
        // then store at the first level whose bit is clear; k == 31 leaves the root, kept in st[0]
        const int ones = (k & 1) ? ((k & 2) ? ((k & 4) ? ((k & 8) ? ((k & 16) ? 5 : 4) : 3) : 2) : 1) : 0;
#pragma unroll
        for (int a = 0; a < SC_RU; ++a)
#pragma unroll
            for (int b = 0; b < SC_RI; ++b) {
                double v = c[a][b];
#pragma unroll
                for (int lev = 0; lev < 5; ++lev)
                    if (lev < ones) v = __dadd_rn(st[lev][a][b], v);
#pragma unroll
                for (int lev = 0; lev < 5; ++lev)
                    if (lev == (ones == 5 ? 0 : ones)) st[lev][a][b] = v;
            }
    }
#pragma unroll
    for (int a = 0; a < SC_RU; ++a) {
        if (r0 + a >= n_rows) break;
        double* out = scores + (size_t)(r0 + a) * ld;
#pragma unroll
        for (int b = 0; b < SC_RI; ++b) {
            const int64_t i = i0 + 32 * b;
            if (i >= n_items) continue;
            const double part = st[0][a][b];
            out[i] = biased ? __dadd_rn(__dadd_rn(hb[r0 + a], bi[i]), part) : part;
        }
    }
}

int mf_score_block_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, int f, int biased, double mu,
                       const double* pu, const double* qi, const double* bu, const double* bi, const double* yj,
                       const int64_t* u_ptr, const int32_t* ui_idx, double* scores, int64_t ld, cudaStream_t st) {
    if (n_rows < 0 || n_items < 0 || f < 0 || ld < n_items || (f > 0 && (!pu || !qi)) || (biased && (!bu || !bi)) ||
        (yj && (!u_ptr || !ui_idx)) || (n_rows > 0 && n_items > 0 && (!rows || !scores))) {
        set_error("mf_score_block: invalid argument");
        return SB2_ERR_INVALID;
    }
    if (n_rows == 0 || n_items == 0) return SB2_OK;
    const int T = (f + 31) / 32;
    DevBuf d_qr, d_pr, d_hb;
    SB2_TRY(d_qr.alloc((size_t)n_items * 32 * T * 8, st));
    SB2_TRY(d_pr.alloc((size_t)n_rows * 32 * T * 8, st));
    SB2_TRY(d_hb.alloc((size_t)n_rows * 8, st));
    const int64_t cap = (int64_t)sm_count() * 16;
    int64_t g = ceil_div((int64_t)n_items * 32 * T, 256);
    top_n_repack_items_kernel<<<(unsigned)std::max<int64_t>(1, std::min(g, cap)), 256, 0, st>>>(
        n_items, f, T, qi, d_qr.as<double>());
    SB2_LAUNCH_CHECK();
    g = ceil_div(n_rows * 32 * std::max(T, 1), 256);
    top_n_repack_users_kernel<<<(unsigned)std::max<int64_t>(1, std::min(g, cap)), 256, 0, st>>>(
        n_rows, rows, f, T, biased, mu, pu, bu, yj, u_ptr, ui_idx, d_pr.as<double>(), d_hb.as<double>());
    SB2_LAUNCH_CHECK();
    const dim3 grid((unsigned)ceil_div(n_items, SC_ITEMS), (unsigned)ceil_div(n_rows, SC_ROWS));
    if (grid.y > 65535u) {
        set_error("mf_score_block: at most %d rows per call", 65535 * SC_ROWS);
        return SB2_ERR_INVALID;
    }
    top_n_score_kernel<<<grid, SC_WARPS * 32, 0, st>>>(n_rows, n_items, T, biased, d_pr.as<double>(),
                                                       d_qr.as<double>(), d_hb.as<double>(), bi, scores, ld);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

// ------------------------------------------------------------------------------------------------
// Selection.  One block per row.  Every candidate (an item the user did not rate: a shared-memory bitmap built
// from ur[u]) gets the value AlgoBase.test gives it -- default_est where impossible == 1, minus the offset,
// np.minimum(high, .) then np.maximum(low, .) -- and the key (order-preserving integer image of that double,
// -0.0 as +0.0, NaN below every number, item id as the tie-break).
// One pass over the row keeps the best K = min(n, SEL_KMAX) candidates: survivors of a running threshold are
// appended to a shared buffer; when it might overflow it is sorted (bitonic) and cut to K, whose last entry
// becomes the threshold.  A final sort emits them.  n > SEL_KMAX runs further passes, each taking the next K
// strictly after the last emitted entry.
// ------------------------------------------------------------------------------------------------
constexpr int SEL_PER = 4;                          // candidates per thread per tile
constexpr int SEL_TILE = SEL_THREADS * SEL_PER;
constexpr int SEL_KMAX = 2048;                      // entries kept per pass

__global__ void __launch_bounds__(SEL_THREADS)
top_n_select_kernel(int64_t n_items, const int32_t* __restrict__ rows, const double* __restrict__ scores, int64_t ld,
                    const uint8_t* __restrict__ impossible, double def, double offset, double low, double high,
                    const int64_t* __restrict__ u_ptr, const int32_t* __restrict__ ui_idx, int n, int cap,
                    int32_t* __restrict__ items_out, double* __restrict__ est_out, int32_t* __restrict__ count_out,
                    int* __restrict__ zero_div) {
    extern __shared__ __align__(16) unsigned long long top_n_smem[];
    unsigned long long* bkey = top_n_smem;                          // [cap]
    int* bitem = reinterpret_cast<int*>(bkey + cap);                // [cap]
    unsigned* rated = reinterpret_cast<unsigned*>(bitem + cap);     // [ceil(n_items / 32)]
    __shared__ int s_cnt;
    const int tid = threadIdx.x;
    const int64_t r = blockIdx.x;
    const int32_t u = rows[r];
    const double* srow = scores + (size_t)r * ld;
    const uint8_t* irow = impossible ? impossible + (size_t)r * ld : nullptr;
    int32_t* iout = items_out + (size_t)r * n;
    double* eout = est_out + (size_t)r * n;
    const int64_t words = (n_items + 31) >> 5;
    for (int64_t x = tid; x < words; x += SEL_THREADS) rated[x] = 0u;
    __syncthreads();
    for (int64_t a = u_ptr[u] + tid; a < u_ptr[u + 1]; a += SEL_THREADS) {
        const int32_t j = ui_idx[a];
        atomicOr(&rated[j >> 5], 1u << (j & 31));
    }
    int emitted = 0;
    bool bounded = false;
    unsigned long long bk = 0ull;
    int bi = 0;
    while (true) {
        const int K = n - emitted < SEL_KMAX ? n - emitted : SEL_KMAX;
        bool thr = false;
        unsigned long long tk = 0ull;
        int ti = 0;
        if (tid == 0) s_cnt = 0;
        __syncthreads();
        for (int64_t i0 = 0; i0 < n_items; i0 += SEL_TILE) {
#pragma unroll
            for (int e = 0; e < SEL_PER; ++e) {
                const int64_t i = i0 + e * SEL_THREADS + tid;
                if (i < n_items && !((rated[i >> 5] >> (i & 31)) & 1u)) {
                    const int code = irow ? irow[i] : 0;
                    if (code == 2 && !bounded) atomicExch(zero_div, 1);
                    const unsigned long long k = top_n_key(top_n_value(srow[i], code, def, offset, low, high));
                    const int ii = (int)i;
                    if ((!bounded || top_n_better(bk, bi, k, ii)) && (!thr || top_n_better(k, ii, tk, ti))) {
                        const int s = atomicAdd(&s_cnt, 1);
                        bkey[s] = k;
                        bitem[s] = ii;
                    }
                }
            }
            __syncthreads();
            const int c = s_cnt;
            if (c > cap - SEL_TILE) {     // the next tile might not fit: keep the best K (c > K here)
                top_n_sort(bkey, bitem, c);
                tk = bkey[K - 1];
                ti = bitem[K - 1];
                thr = true;
                __syncthreads();
                if (tid == 0) s_cnt = K;
            }
            __syncthreads();
        }
        const int c = s_cnt;
        top_n_sort(bkey, bitem, c);
        const int m = c < K ? c : K;
        for (int j = tid; j < m; j += SEL_THREADS) {
            const int it = bitem[j];
            iout[emitted + j] = it;
            eout[emitted + j] = top_n_value(srow[it], irow ? irow[it] : 0, def, offset, low, high);
        }
        emitted += m;
        if (m < K || emitted >= n) break;
        bk = bkey[m - 1];
        bi = bitem[m - 1];
        bounded = true;
        __syncthreads();
    }
    for (int j = emitted + tid; j < n; j += SEL_THREADS) {
        iout[j] = -1;
        eout[j] = __longlong_as_double(0x7FF8000000000000ll);
    }
    if (tid == 0) count_out[r] = emitted;
}

int top_n_select_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                     const uint8_t* impossible, double default_est, double offset, double low, double high,
                     const int64_t* u_ptr, const int32_t* ui_idx, int n, int32_t* items_out, double* est_out,
                     int32_t* count_out, cudaStream_t st) {
    if (n < 1) {
        set_error("top_n_select: n must be >= 1 (got %d)", n);
        return SB2_ERR_INVALID;
    }
    if (n_rows < 0 || n_items < 0 || n_items > 0x7FFFFFFF || ld < n_items ||
        (n_rows > 0 && (!rows || !scores || !u_ptr || !ui_idx || !items_out || !est_out || !count_out))) {
        set_error("top_n_select: invalid argument");
        return SB2_ERR_INVALID;
    }
    if (n_rows == 0) return SB2_OK;
    const int k0 = n < SEL_KMAX ? n : SEL_KMAX;
    int cap = 1;
    while (cap < k0 + SEL_TILE || cap < 2 * k0) cap <<= 1;
    const size_t smem = (size_t)cap * 12 + (size_t)((n_items + 31) >> 5) * 4;
    int dev = 0, max_smem = 0;
    SB2_CUDA(cudaGetDevice(&dev));
    SB2_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (smem + 64 > (size_t)max_smem) {
        set_error("top_n_select: %lld items need a %zu-byte rated-item bitmap, beyond shared memory",
                  (long long)n_items, smem);
        return SB2_ERR_UNSUPPORTED;
    }
    SB2_CUDA(cudaFuncSetAttribute(top_n_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DevBuf d_flag;
    if (impossible) {
        SB2_TRY(d_flag.alloc(sizeof(int), st));
        SB2_CUDA(cudaMemsetAsync(d_flag.p, 0, sizeof(int), st));
    }
    if (n_rows > 0x7FFFFFFF) {
        set_error("top_n_select: too many rows");
        return SB2_ERR_INVALID;
    }
    top_n_select_kernel<<<(unsigned)n_rows, SEL_THREADS, smem, st>>>(n_items, rows, scores, ld, impossible, default_est,
                                                                      offset, low, high, u_ptr, ui_idx, n, cap,
                                                                      items_out, est_out, count_out,
                                                                      d_flag.as<int>());
    SB2_LAUNCH_CHECK();
    if (impossible) {
        int flag = 0;
        SB2_CUDA(cudaMemcpyAsync(&flag, d_flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        SB2_CUDA(cudaStreamSynchronize(st));
        if (flag) {
            set_error("division by zero");
            return SB2_ERR_ZERO_DIVISION;
        }
    }
    return SB2_OK;
}

}  // namespace sb2
