// Hits of top-N lists against held-out relevant items, and the coverage / novelty / diversity of the lists themselves:
// the per-user values behind AlgoBase.top_n_measures and AlgoBase.top_n_list_measures.
//
// Hits (accuracy.top_n_measures is the definition; DESIGN.md section 3.9).
// Input: one block of sb2_top_n_select_dev's output (items [rows, ld], count [rows]), a cutoff w <= ld, and per row
// the sorted distinct relevant inner item ids rel_idx[rel_ptr[b], rel_ptr[b + 1]).  For every row b:
//   H_b  = {p < min(count[b], w) : items[b, p] in the row's relevant list}
//   hits = |H_b|,  rr = sum of inv[p] over H_b,  dcg = sum of disc[p] over H_b
// with the sums taken in ascending p from +0.0, one plain fp64 add at a time: the definition's order.  inv and disc
// are the host's tables (no log2 on the device), so the values carry the host's bits.
//
// One warp per row.  Lane l tests positions p = l, l + 32, ... by binary search in the row's list, the warp ballots
// each 32-position chunk, and every lane walks the chunk's hits in ascending p, taking inv[p] / disc[p] from the
// lane that loaded them; the sums are therefore warp-uniform and lane 0 stores them.
#include "common.cuh"

namespace sb2 {

constexpr int TE_THREADS = 256;
constexpr int TE_ROWS = TE_THREADS / 32;    // rows per CTA

__global__ void __launch_bounds__(TE_THREADS)
top_n_hits_kernel(int64_t n_rows, const int32_t* __restrict__ items, int64_t ld, const int32_t* __restrict__ count,
                  int w, const int64_t* __restrict__ rel_ptr, const int32_t* __restrict__ rel_idx, int64_t rel_len,
                  const double* __restrict__ inv, const double* __restrict__ disc, int32_t* __restrict__ hits,
                  double* __restrict__ rr, double* __restrict__ dcg, int* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * TE_ROWS + (threadIdx.x >> 5);
    if (b >= n_rows) return;
    // offsets check: 0 <= rel_ptr[b] <= rel_ptr[b + 1] <= rel_len, and the row's list strictly ascending
    int64_t lo = rel_ptr[b], hi = rel_ptr[b + 1];
    bool ok = 0 <= lo && lo <= hi && hi <= rel_len;
    lo = lo < 0 ? 0 : (lo > rel_len ? rel_len : lo);
    hi = hi < lo ? lo : (hi > rel_len ? rel_len : hi);
    for (int64_t j = lo + 1 + lane; j < hi; j += 32) ok = ok && rel_idx[j - 1] < rel_idx[j];
    if (!ok) atomicExch(bad, 1);

    int c = count[b];
    c = c < 0 ? 0 : (c < w ? c : w);
    const int32_t* row = items + b * ld;
    int h = 0;
    double a = 0.0, d = 0.0;
    for (int p0 = 0; p0 < c; p0 += 32) {
        const int p = p0 + lane;
        bool hit = false;
        double x_inv = 0.0, x_disc = 0.0;
        if (p < c) {
            const int32_t it = row[p];
            int64_t l = lo, r = hi;     // first entry >= it in [lo, hi)
            while (l < r) {
                const int64_t mid = l + ((r - l) >> 1);
                if (rel_idx[mid] < it) l = mid + 1;
                else r = mid;
            }
            hit = l < hi && rel_idx[l] == it;
            if (hit) {
                x_inv = inv[p];
                x_disc = disc[p];
            }
        }
        unsigned mask = __ballot_sync(0xFFFFFFFFu, hit);
        h += __popc(mask);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            a = __dadd_rn(a, __shfl_sync(0xFFFFFFFFu, x_inv, src));
            d = __dadd_rn(d, __shfl_sync(0xFFFFFFFFu, x_disc, src));
        }
    }
    if (lane == 0) {
        hits[b] = h;
        rr[b] = a;
        dcg[b] = d;
    }
}

int top_n_hits_dev(int64_t n_rows, const int32_t* items, int64_t ld, const int32_t* count, int w,
                   const int64_t* rel_ptr, const int32_t* rel_idx, int64_t rel_len, const double* inv,
                   const double* disc, int32_t* hits, double* rr, double* dcg, cudaStream_t st) {
    if (n_rows < 0 || w < 0 || ld < w || rel_len < 0 || (rel_len > 0 && !rel_idx) ||
        (n_rows > 0 && (!items || !count || !rel_ptr || !hits || !rr || !dcg || (w > 0 && (!inv || !disc))))) {
        set_error("top_n_hits: invalid argument");
        return SB2_ERR_INVALID;
    }
    if (n_rows == 0) return SB2_OK;
    const int64_t blocks = ceil_div(n_rows, TE_ROWS);
    if (blocks > 0x7FFFFFFF) {
        set_error("top_n_hits: too many rows");
        return SB2_ERR_INVALID;
    }
    DevBuf d_bad;
    SB2_TRY(d_bad.alloc(sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(d_bad.p, 0, sizeof(int), st));
    top_n_hits_kernel<<<(unsigned)blocks, TE_THREADS, 0, st>>>(n_rows, items, ld, count, w, rel_ptr, rel_idx, rel_len,
                                                              inv, disc, hits, rr, dcg, d_bad.as<int>());
    SB2_LAUNCH_CHECK();
    int bad = 0;
    SB2_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (bad) {
        set_error("top_n_hits: malformed relevant lists (need 0 <= rel_ptr[b] <= rel_ptr[b + 1] <= rel_len and each "
                  "list strictly ascending)");
        return SB2_ERR_INVALID;
    }
    return SB2_OK;
}

// Coverage, novelty and intra-list similarity of top-N lists: the per-user values behind AlgoBase.top_n_list_measures
// (accuracy.top_n_list_measures is the definition; DESIGN.md section 3.11).  For row b with c = min(count[b], w) and
// L = items[b, 0 .. c):
//   covered = some p < c has est[b, p] >= threshold (any p < c without a threshold; a NaN est never passes),
//   nov     = the sum of info[L[p]] over p ascending,
//   ils     = the sum of sim[L[p], L[q]] over p < q, p ascending and q ascending inside it,
// each sum from +0.0 with one plain fp64 add per term, and seen[L[p]] = 1 for every p.
//
// One warp per row.  Lane l gathers the terms of positions l, l + 32, ... of a 32-wide chunk and every lane folds the
// chunk in ascending position by shuffle, so the sums are warp-uniform and lane 0 stores them.  An item outside
// [0, n_items) sets *bad and reads (and marks) nothing.
__global__ void __launch_bounds__(TE_THREADS)
top_n_lists_kernel(int64_t n_rows, const int32_t* __restrict__ items, int64_t ld, const double* __restrict__ est,
                   const int32_t* __restrict__ count, int w, int has_threshold, double threshold, int64_t n_items,
                   const double* __restrict__ info, const double* __restrict__ sim, int32_t* __restrict__ covered,
                   double* __restrict__ nov, double* __restrict__ ils, uint8_t* __restrict__ seen,
                   int* __restrict__ bad) {
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * TE_ROWS + (threadIdx.x >> 5);
    if (b >= n_rows) return;
    int c = count[b];
    c = c < 0 ? 0 : (c < w ? c : w);
    const int32_t* row = items + b * ld;
    bool ok = true, cov = false;
    double s = 0.0;
    for (int p0 = 0; p0 < c; p0 += 32) {
        const int p = p0 + lane;
        double x = 0.0;
        if (p < c) {
            const int32_t it = row[p];
            if (0 <= it && it < n_items) {
                x = info[it];
                seen[it] = 1;
            } else {
                ok = false;
            }
            cov = cov || !has_threshold || est[b * ld + p] >= threshold;
        }
        const int m = c - p0 < 32 ? c - p0 : 32;
        for (int j = 0; j < m; ++j) s = __dadd_rn(s, __shfl_sync(0xFFFFFFFFu, x, j));
    }
    cov = __any_sync(0xFFFFFFFFu, cov);
    if (!__all_sync(0xFFFFFFFFu, ok)) {
        if (lane == 0) atomicExch(bad, 1);
        return;
    }
    double t = 0.0;
    if (sim) {
        for (int p = 0; p + 1 < c; ++p) {
            const double* srow = sim + (int64_t)row[p] * n_items;
            for (int q0 = p + 1; q0 < c; q0 += 32) {
                const int q = q0 + lane;
                const double y = q < c ? srow[row[q]] : 0.0;
                const int m = c - q0 < 32 ? c - q0 : 32;
                for (int j = 0; j < m; ++j) t = __dadd_rn(t, __shfl_sync(0xFFFFFFFFu, y, j));
            }
        }
    }
    if (lane == 0) {
        covered[b] = cov ? 1 : 0;
        nov[b] = s;
        if (sim) ils[b] = t;
    }
}

int top_n_lists_dev(int64_t n_rows, const int32_t* items, int64_t ld, const double* est, const int32_t* count, int w,
                    int has_threshold, double threshold, int64_t n_items, const double* info, const double* sim,
                    int32_t* covered, double* nov, double* ils, uint8_t* seen, cudaStream_t st) {
    if (n_rows < 0 || w < 0 || ld < w || n_items < 0 || n_items > 0x7FFFFFFF ||
        (n_rows > 0 && (!items || !count || !covered || !nov || (has_threshold && !est) || (sim && !ils) ||
                        (w > 0 && n_items > 0 && (!info || !seen))))) {
        set_error("top_n_lists: invalid argument");
        return SB2_ERR_INVALID;
    }
    if (n_rows == 0) return SB2_OK;
    const int64_t blocks = ceil_div(n_rows, TE_ROWS);
    if (blocks > 0x7FFFFFFF) {
        set_error("top_n_lists: too many rows");
        return SB2_ERR_INVALID;
    }
    DevBuf d_bad;
    SB2_TRY(d_bad.alloc(sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(d_bad.p, 0, sizeof(int), st));
    top_n_lists_kernel<<<(unsigned)blocks, TE_THREADS, 0, st>>>(n_rows, items, ld, est, count, w, has_threshold,
                                                               threshold, n_items, info, sim, covered, nov, ils, seen,
                                                               d_bad.as<int>());
    SB2_LAUNCH_CHECK();
    int bad = 0;
    SB2_CUDA(cudaMemcpyAsync(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (bad) {
        set_error("top_n_lists: a listed item is outside [0, n_items)");
        return SB2_ERR_INVALID;
    }
    return SB2_OK;
}

}  // namespace sb2
