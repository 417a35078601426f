// Hits of top-N lists against held-out relevant items, the coverage / novelty / diversity of the lists themselves, and
// where the held-out items rank among all candidates: the per-user values behind AlgoBase.top_n_measures,
// AlgoBase.top_n_list_measures and AlgoBase.rank_measures.
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
#include "top_n.cuh"

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

// Where the held-out items land in each user's whole ranking: the per-user counts behind AlgoBase.rank_measures
// (accuracy.rank_measures is the definition; DESIGN.md section 3.12).  Input: one block of scores exactly as
// sb2_top_n_select_dev receives it, and per row the sorted distinct relevant inner item ids rel_idx[rel_ptr[b],
// rel_ptr[b + 1]).  The candidates of row b are the items its user did not rate, ordered as the selection orders them
// (top_n.cuh); a relevant candidate's position is the number of candidates that rank before it.  For every row:
//   c = the number of candidates, k = the number of relevant candidates, s = the sum of their positions and f the
//   smallest one (-1 when k = 0).
//
// One CTA per row.  The relevant candidates are loaded RK_TILE at a time into shared memory and sorted best-first;
// one pass over the row's scores then gives each candidate x the number q of tile entries at least as good as x (a
// binary search).  x ranks before exactly the m - q entries after those, so the tile's position sum is the sum of
// m - q over the candidates, and its best entry's position the number of candidates with q = 0.  Everything is an
// integer count, so nothing depends on the launch geometry.
constexpr int RK_TILE = 2048;     // relevant candidates per pass; a power of two, which top_n_sort pads to

__device__ __forceinline__ long long rk_block_sum(long long v, long long* red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    __syncthreads();     // the previous sum's readers are done with red
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    long long t = 0;
#pragma unroll
    for (int w = 0; w < SEL_THREADS / 32; ++w) t += red[w];
    return t;
}

__global__ void __launch_bounds__(SEL_THREADS)
top_n_ranks_kernel(int64_t n_items, const int32_t* __restrict__ rows, const double* __restrict__ scores, int64_t ld,
                   const uint8_t* __restrict__ impossible, double def, double offset, double low, double high,
                   const int64_t* __restrict__ u_ptr, const int32_t* __restrict__ ui_idx,
                   const int64_t* __restrict__ rel_ptr, const int32_t* __restrict__ rel_idx, int64_t rel_len,
                   int32_t* __restrict__ c_out, int32_t* __restrict__ k_out, int64_t* __restrict__ s_out,
                   int32_t* __restrict__ f_out, int* __restrict__ flags) {
    extern __shared__ __align__(16) unsigned long long top_n_rank_smem[];
    unsigned long long* tkey = top_n_rank_smem;                      // [RK_TILE]
    int* titem = reinterpret_cast<int*>(tkey + RK_TILE);             // [RK_TILE]
    unsigned* rated = reinterpret_cast<unsigned*>(titem + RK_TILE);  // [ceil(n_items / 32)]
    __shared__ long long red[SEL_THREADS / 32];
    __shared__ int s_m;
    const int tid = threadIdx.x;
    const int64_t r = blockIdx.x;
    const int32_t u = rows[r];
    const double* srow = scores + (size_t)r * ld;
    const uint8_t* irow = impossible ? impossible + (size_t)r * ld : nullptr;
    const int64_t words = (n_items + 31) >> 5;
    for (int64_t x = tid; x < words; x += SEL_THREADS) rated[x] = 0u;
    __syncthreads();
    for (int64_t a = u_ptr[u] + tid; a < u_ptr[u + 1]; a += SEL_THREADS) {
        const int32_t j = ui_idx[a];
        atomicOr(&rated[j >> 5], 1u << (j & 31));
    }
    // offsets check: 0 <= rel_ptr[b] <= rel_ptr[b + 1] <= rel_len, and the row's list strictly ascending inside
    // [0, n_items); a row that fails it reads nothing more
    int64_t lo = rel_ptr[r], hi = rel_ptr[r + 1];
    bool ok = 0 <= lo && lo <= hi && hi <= rel_len;
    lo = lo < 0 ? 0 : (lo > rel_len ? rel_len : lo);
    hi = hi < lo ? lo : (hi > rel_len ? rel_len : hi);
    for (int64_t j = lo + tid; j < hi; j += SEL_THREADS) {
        const int32_t it = rel_idx[j];
        ok = ok && 0 <= it && it < n_items && (j == lo || rel_idx[j - 1] < it);
    }
    if (__syncthreads_or(!ok)) {      // also orders the bitmap before its reads
        if (tid == 0) atomicExch(&flags[1], 1);
        return;
    }
    int cnt = 0, k = 0, f = -1;
    long long s = 0;
    for (int64_t t0 = lo;; t0 += RK_TILE) {
        const bool first = t0 == lo;
        const int64_t t1 = hi - t0 < RK_TILE ? hi : t0 + RK_TILE;
        if (tid == 0) s_m = 0;
        __syncthreads();
        for (int64_t j = t0 + tid; j < t1; j += SEL_THREADS) {
            const int32_t it = rel_idx[j];
            if (!((rated[it >> 5] >> (it & 31)) & 1u)) {
                const int q = atomicAdd(&s_m, 1);
                tkey[q] = top_n_key(top_n_value(srow[it], irow ? irow[it] : 0, def, offset, low, high));
                titem[q] = it;
            }
        }
        __syncthreads();
        const int m = s_m;
        if (m > 0) top_n_sort(tkey, titem, m);
        if (first || m > 0) {
            long long below = 0;
            int above = 0, c_loc = 0;
            for (int64_t i = tid; i < n_items; i += SEL_THREADS) {
                if ((rated[i >> 5] >> (i & 31)) & 1u) continue;
                const int code = irow ? irow[i] : 0;
                if (first) {
                    ++c_loc;
                    if (code == 2) atomicExch(&flags[0], 1);
                }
                if (m > 0) {
                    const unsigned long long key = top_n_key(top_n_value(srow[i], code, def, offset, low, high));
                    int l = 0, h = m;        // l = the number of tile entries at least as good as (key, i)
                    while (l < h) {
                        const int mid = (l + h) >> 1;
                        if (top_n_better(key, (int)i, tkey[mid], titem[mid])) h = mid;
                        else l = mid + 1;
                    }
                    below += m - l;
                    above += l == 0;
                }
            }
            if (first) cnt = (int)rk_block_sum(c_loc, red);
            if (m > 0) {
                s += rk_block_sum(below, red);
                const int pos = (int)rk_block_sum(above, red);
                f = f < 0 || pos < f ? pos : f;
                k += m;
            }
        }
        if (t1 >= hi) break;
        __syncthreads();     // every thread is done with the tile before it is reloaded
    }
    if (tid == 0) {
        c_out[r] = cnt;
        k_out[r] = k;
        s_out[r] = s;
        f_out[r] = f;
    }
}

int top_n_ranks_dev(int64_t n_rows, const int32_t* rows, int64_t n_items, const double* scores, int64_t ld,
                    const uint8_t* impossible, double default_est, double offset, double low, double high,
                    const int64_t* u_ptr, const int32_t* ui_idx, const int64_t* rel_ptr, const int32_t* rel_idx,
                    int64_t rel_len, int32_t* c, int32_t* k, int64_t* s, int32_t* f, cudaStream_t st) {
    if (n_rows < 0 || n_items < 0 || n_items > 0x7FFFFFFF || ld < n_items || rel_len < 0 ||
        (rel_len > 0 && !rel_idx) ||
        (n_rows > 0 && (!rows || !scores || !u_ptr || !ui_idx || !rel_ptr || !c || !k || !s || !f))) {
        set_error("top_n_ranks: invalid argument");
        return SB2_ERR_INVALID;
    }
    if (n_rows == 0) return SB2_OK;
    if (n_rows > 0x7FFFFFFF) {
        set_error("top_n_ranks: too many rows");
        return SB2_ERR_INVALID;
    }
    const size_t smem = (size_t)RK_TILE * 12 + (size_t)((n_items + 31) >> 5) * 4;
    int dev = 0, max_smem = 0;
    SB2_CUDA(cudaGetDevice(&dev));
    SB2_CUDA(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (smem + 64 + 8 * (SEL_THREADS / 32) > (size_t)max_smem) {
        set_error("top_n_ranks: %lld items need a %zu-byte rated-item bitmap, beyond shared memory",
                  (long long)n_items, smem);
        return SB2_ERR_UNSUPPORTED;
    }
    SB2_CUDA(cudaFuncSetAttribute(top_n_ranks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DevBuf d_flags;
    SB2_TRY(d_flags.alloc(2 * sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(d_flags.p, 0, 2 * sizeof(int), st));
    top_n_ranks_kernel<<<(unsigned)n_rows, SEL_THREADS, smem, st>>>(n_items, rows, scores, ld, impossible, default_est,
                                                                     offset, low, high, u_ptr, ui_idx, rel_ptr,
                                                                     rel_idx, rel_len, c, k, s, f,
                                                                     d_flags.as<int>());
    SB2_LAUNCH_CHECK();
    int flags[2] = {0, 0};
    SB2_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof(flags), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (flags[1]) {
        set_error("top_n_ranks: malformed relevant lists (need 0 <= rel_ptr[b] <= rel_ptr[b + 1] <= rel_len and each "
                  "list strictly ascending inside [0, n_items))");
        return SB2_ERR_INVALID;
    }
    if (flags[0]) {
        set_error("division by zero");
        return SB2_ERR_ZERO_DIVISION;
    }
    return SB2_OK;
}

}  // namespace sb2
