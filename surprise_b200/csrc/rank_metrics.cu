// Per-user integer counts behind accuracy.fcp and accuracy.precision_recall_at_k (DESIGN.md section 3.7).
//
// Input: a segment CSR over the predictions (seg_ptr, one segment per user, entries in prediction order) with the
// true ratings r and the estimates est in fp64.  One kernel serves both metrics:
//   fcp mode       for every row j: nc += #{i : e_j > e_i and r_j > r_i}, nd += #{i : e_j >= e_i and r_j < r_i}
//   precision mode for every row j: rank_j = #{i : e_i > e_j} + #{i < j : e_i == e_j} (only where 0 < k_eff < m);
//                  top_j = rank_j < k_eff; n_rel += r_j >= t, n_rec += top_j and e_j >= t, n_rr += that and r_j >= t
// with i running over j's own segment.  Compares are fp64, so NaN compares false and -0.0 == +0.0, as in Python.
//
// Work item = 256 consecutive rows (one per thread).  The CTA streams the entries of every segment its rows touch
// through a shared-memory tile; each thread compares its row with the tile entries of its own segment.  A user longer
// than 256 rows therefore spans several CTAs, each re-reading the whole segment (from L2), and short users share one.
// Threads count in registers; the CTA reduces per user and issues one 64-bit integer atomicAdd per counter per user,
// so the counts do not depend on the launch geometry or on the order of the atomics.
#include "common.cuh"

namespace sb2 {

constexpr int RM_THREADS = 256;     // rows per work item
constexpr int RM_WARPS = RM_THREADS / 32;
constexpr int RM_TILE = 1024;       // segment entries per shared-memory tile

// last s in [lo, hi) with seg_ptr[s] <= j (lo when there is none); seg_ptr need not be sorted for this to stay in range
__device__ __forceinline__ int64_t rm_segment_of(const int64_t* __restrict__ seg_ptr, int64_t lo, int64_t hi,
                                                 int64_t j) {
    while (hi - lo > 1) {
        const int64_t mid = lo + ((hi - lo) >> 1);
        if (seg_ptr[mid] <= j) lo = mid;
        else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ int64_t rm_clamp(int64_t x, int64_t n) { return x < 0 ? 0 : (x > n ? n : x); }

// NC counters per segment: 2 in fcp mode (nc, nd), 3 in precision mode (n_rel, n_rec, n_rr)
template <int NC>
__global__ void __launch_bounds__(RM_THREADS, 4)
rank_metrics_kernel(int64_t n_seg, int64_t n, const int64_t* __restrict__ seg_ptr, const double* __restrict__ r,
                    const double* __restrict__ est, const int64_t* __restrict__ k_eff, double threshold,
                    unsigned long long* __restrict__ counts, int* __restrict__ bad) {
    constexpr bool FCP = NC == 2;
    __shared__ double2 tile[RM_TILE];                       // (est, r)
    __shared__ unsigned long long acc[NC][RM_THREADS];      // per run of equal segments in the CTA
    __shared__ int64_t row_seg[RM_THREADS];
    __shared__ int64_t run_seg[RM_THREADS];
    __shared__ int64_t span[2];
    __shared__ int warp_runs[RM_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // offsets check: seg_ptr[0] == 0, non-decreasing, seg_ptr[n_seg] == n (every read below is clamped regardless)
    for (int64_t s = (int64_t)blockIdx.x * RM_THREADS + tid; s <= n_seg; s += (int64_t)gridDim.x * RM_THREADS) {
        const int64_t p = seg_ptr[s];
        bool ok = s == 0 ? p == 0 : seg_ptr[s - 1] <= p;
        if (s == n_seg) ok = ok && p == n;
        if (!ok) atomicExch(bad, 1);
    }
    const int64_t row0 = (int64_t)blockIdx.x * RM_THREADS;
    if (row0 >= n) return;
    const int64_t rows = n - row0 < RM_THREADS ? n - row0 : RM_THREADS;
    if (tid == 0) {
        span[0] = rm_segment_of(seg_ptr, 0, n_seg, row0);
        span[1] = rm_segment_of(seg_ptr, 0, n_seg, row0 + rows - 1);
    }
    __syncthreads();
    const int64_t s0 = span[0], s1 = span[1] < s0 ? s0 : span[1];
    const int64_t c_lo = rm_clamp(seg_ptr[s0], n);
    int64_t c_hi = rm_clamp(seg_ptr[s1 + 1], n);
    c_hi = c_hi < c_lo ? c_lo : c_hi;

    const bool active = tid < rows;
    const int64_t j = row0 + tid;
    const int64_t s = active ? rm_segment_of(seg_ptr, s0, s1 + 1, j) : -1;
    int64_t lo = 0, hi = 0;
    double ej = 0.0, rj = 0.0;
    if (active) {
        lo = rm_clamp(seg_ptr[s], n);
        hi = rm_clamp(seg_ptr[s + 1], n);
        ej = est[j];
        rj = r[j];
    }
    // fcp: c0 = nc, c1 = nd.  precision: c0 = rank
    unsigned long long c0 = 0, c1 = 0;
    int64_t kk = 0;
    bool scan = active;
    if constexpr (!FCP) {
        if (active) {
            kk = k_eff[s];
            scan = kk > 0 && kk < hi - lo;
        }
    }
    if (__syncthreads_or(scan)) {
        for (int64_t t0 = c_lo; t0 < c_hi; t0 += RM_TILE) {
            const int cnt = (int)(c_hi - t0 < RM_TILE ? c_hi - t0 : RM_TILE);
            for (int x = tid; x < cnt; x += RM_THREADS) tile[x] = make_double2(est[t0 + x], r[t0 + x]);
            __syncthreads();
            int a = 0, b = 0;     // this row's entries in the tile: [a, b)
            if (scan) {
                const int64_t a64 = (lo > t0 ? lo : t0) - t0, b64 = (hi < t0 + cnt ? hi : t0 + cnt) - t0;
                a = (int)(a64 < cnt ? a64 : cnt);
                b = (int)(b64 > 0 ? b64 : 0);
            }
            unsigned u0 = 0, u1 = 0;
            if constexpr (FCP) {
#pragma unroll 4
                for (int x = a; x < b; ++x) {
                    const double2 v = tile[x];
                    u0 += (ej > v.x) & (rj > v.y);
                    u1 += (ej >= v.x) & (rj < v.y);
                }
            } else {
                // entries before j in this tile are x < self
                const int self = j < t0 ? 0 : (j - t0 < cnt ? (int)(j - t0) : cnt);
#pragma unroll 4
                for (int x = a; x < b; ++x) {
                    const double e = tile[x].x;
                    u0 += (e > ej) | ((e == ej) & (x < self));
                }
            }
            c0 += u0;
            c1 += u1;
            __syncthreads();
        }
    }
    unsigned long long v[NC];
    if constexpr (FCP) {
        v[0] = c0;
        v[1] = c1;
    } else {
        const bool top = kk >= hi - lo || (int64_t)c0 < kk;   // kk >= m: every row, kk <= 0: none (c0 >= 0)
        const bool rel = rj >= threshold;
        const bool rec = active && top && ej >= threshold;
        v[0] = active && rel;
        v[1] = rec;
        v[2] = rec && rel;
    }

    // CTA reduction: rows are sorted by segment, so each segment's rows form one run
    row_seg[tid] = s;
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[c][tid] = 0ull;
    __syncthreads();
    const bool head = active && (tid == 0 || row_seg[tid - 1] != s);
    const unsigned heads = __ballot_sync(0xFFFFFFFFu, head);
    if (lane == 0) warp_runs[warp] = __popc(heads);
    __syncthreads();
    int run = __popc(heads & (0xFFFFFFFFu >> (31 - lane))) - 1, n_runs = 0;
    for (int w = 0; w < RM_WARPS; ++w) {
        run += w < warp ? warp_runs[w] : 0;
        n_runs += warp_runs[w];
    }
    if (head) run_seg[run] = s;
    // segmented suffix sums inside the warp: the first lane of each run ends up with the run's warp total
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int64_t so = __shfl_down_sync(0xFFFFFFFFu, s, o);
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const unsigned long long x = __shfl_down_sync(0xFFFFFFFFu, v[c], o);
            if (lane + o < 32 && so == s) v[c] += x;
        }
    }
    const int64_t s_prev = __shfl_up_sync(0xFFFFFFFFu, s, 1);
    if (active && (lane == 0 || s_prev != s)) {
#pragma unroll
        for (int c = 0; c < NC; ++c)
            if (v[c]) atomicAdd(&acc[c][run], v[c]);
    }
    __syncthreads();
    if (tid < n_runs) {
#pragma unroll
        for (int c = 0; c < NC; ++c)
            if (acc[c][tid]) atomicAdd(&counts[run_seg[tid] * NC + c], acc[c][tid]);
    }
}

static int rank_metrics_dev(const char* what, int nc, int64_t n_seg, int64_t n, const int64_t* seg_ptr,
                            const double* r, const double* est, const int64_t* k_eff, double threshold,
                            int64_t* counts, cudaStream_t st) {
    if (n_seg < 0 || n < 0 || (n > 0 && n_seg == 0) || !seg_ptr || (n > 0 && (!r || !est)) ||
        (n_seg > 0 && !counts) || (nc == 3 && n_seg > 0 && !k_eff)) {
        set_error("%s: invalid argument", what);
        return SB2_ERR_INVALID;
    }
    if (n_seg > 0) SB2_CUDA(cudaMemsetAsync(counts, 0, (size_t)n_seg * nc * sizeof(int64_t), st));
    DevBuf d_bad;
    SB2_TRY(d_bad.alloc(sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(d_bad.p, 0, sizeof(int), st));
    const int64_t blocks = ceil_div(n > n_seg + 1 ? n : n_seg + 1, RM_THREADS);
    if (blocks > 0x7FFFFFFF) {
        set_error("%s: too many predictions", what);
        return SB2_ERR_INVALID;
    }
    auto* out = reinterpret_cast<unsigned long long*>(counts);
    if (nc == 2)
        rank_metrics_kernel<2><<<(unsigned)blocks, RM_THREADS, 0, st>>>(n_seg, n, seg_ptr, r, est, k_eff, threshold,
                                                                        out, d_bad.as<int>());
    else
        rank_metrics_kernel<3><<<(unsigned)blocks, RM_THREADS, 0, st>>>(n_seg, n, seg_ptr, r, est, k_eff, threshold,
                                                                        out, d_bad.as<int>());
    SB2_LAUNCH_CHECK();
    int bad = 0;
    SB2_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (bad) {
        set_error("%s: malformed segment offsets (need seg_ptr[0] == 0, non-decreasing, seg_ptr[n_seg] == n)", what);
        return SB2_ERR_INVALID;
    }
    return SB2_OK;
}

int fcp_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r, const double* est,
                   int64_t* counts, cudaStream_t st) {
    return rank_metrics_dev("fcp_counts", 2, n_seg, n, seg_ptr, r, est, nullptr, 0.0, counts, st);
}

int precision_at_k_counts_dev(int64_t n_seg, int64_t n, const int64_t* seg_ptr, const double* r, const double* est,
                              const int64_t* k_eff, double threshold, int64_t* counts, cudaStream_t st) {
    return rank_metrics_dev("precision_at_k_counts", 3, n_seg, n, seg_ptr, r, est, k_eff, threshold, counts, st);
}

}  // namespace sb2
