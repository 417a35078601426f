// General similarity path: ARBITRARY double ratings (not on a 1/d grid, negative, huge dynamic range) and duplicate
// (x, y) pairs -- everything the reference's similarities.pyx accepts and the dense integer-digit panels of sim.cu
// cannot represent.  Replaces the same four functions (cosine :28-97, msd :100-166, pearson :169-258,
// pearson_baseline :261-361) on the CUDA cores, in fp64, and in the REFERENCE'S OWN SUMMATION ORDER:
//
//   reference:  for y: for (xi, ri) in yr[y]: for (xj, rj) in yr[y]:  acc[xi, xj] += f(ri, rj)
//
// so for a fixed pair (xi, xj) the additions happen in order of (y, position of the xi entry, position of the xj
// entry).  Here one CTA owns output row xi: it walks xi's entries in (y, position) order -- the x-major transpose of
// the yr CSR, built by a STABLE sort by x -- and for each of them lets its threads sweep yr[y], thread per entry, each
// adding into the row accumulator of its own xj (no two threads of a sweep share an xj: duplicates of one (x, y) are
// split into rounds by their occurrence index).  Every accumulator therefore receives exactly the reference's sequence
// of round-to-nearest products and sums (no FMA contraction), and the per-row finalize applies the reference's
// formula with the reference's operation order: the result is bit-identical to the reference for any input, which
// the tests check against the oracle (and, through it, against the compiled reference's goldens).
// Rows are independent, so a row range [row_begin, row_end) is a shard of a multi-rank build as it stands, and a list
// of rows in any order (sb2_sim_build_rows_dev) is the same rows built by CTAs that look their row up.
//
// Cost: sum_y |yr[y]|^2 pair visits of ~6 L2-resident read-modify-writes each (accumulators: 44 B per column per
// CTA), i.e. HBM/L2-latency work, not tensor work: ~10^2..10^3 x slower than the digit path per build and still
// 10^2..10^3 x faster than the reference.  It is the fallback, chosen only when the ratings leave the grid.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "common.cuh"

namespace sb2 {

enum { G_ST_BAD = 0, G_ST_ZERODIV = 1, G_ST_MAXOCC = 2, G_ST_NWORDS = 4 };

struct GenArgs {
    int64_t n_x, n_y, nnz;
    const int64_t* y_ptr;
    const int32_t* x_idx;
    const double* r;
    const int64_t* x_ptr;   // x-major transpose: entries of x are x_ent[x_ptr[x] .. x_ptr[x + 1]) in (y, position) order
    const int* x_ent;       // entry positions in the yr CSR
    const int* y_of;        // yr segment of every entry
    const uint8_t* occ;     // occurrence index of the entry among the entries with the same (x, y)
    int max_occ;
    // x-major sweep descriptors (no duplicated pairs): for the p-th entry of the x-major order, the yr segment it
    // lies in [xm_b, xm_b + xm_len) and its value
    const int64_t* xm_b;
    const int* xm_len;
    const double* xm_r;     // the row entry's value (rating, or deviation for pearson_baseline)
    const double* val;      // per entry of the yr CSR: the rating, or (pearson_baseline) its deviation
    int min_support;
    double mu, shrinkage;
    const double* bx;
    const double* by;
    int64_t row_begin, n_rows;  // output row b is matrix row rows[b], or row_begin + b when rows is null
    const int32_t* rows;
    int64_t col_begin;      // columns below it are neither accumulated nor written (shard of a symmetric build: the
                            // transposes of the blocks owned by the shards before this one, filled in by the exchange)
    double* sim;            // n_rows x out_ld
    int64_t out_ld;
    double* scratch;        // per CTA: one record per column, [prods | sqi | sqj | freq] (32 B: one sector per
                            // co-rating) or [prods | sqi | sqj | si | sj | freq] for pearson
    int64_t scratch_stride; // doubles per CTA
    int* status;
};

__global__ void gen_entry_kernel(int64_t nnz, int64_t n_x, int64_t n_y, const int64_t* __restrict__ y_ptr,
                                 const int32_t* __restrict__ x_idx, int* __restrict__ y_of, int* __restrict__ ent,
                                 unsigned long long* __restrict__ cnt, int* status) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= nnz) return;
    int64_t lo = 0, hi = n_y;  // largest s with y_ptr[s] <= t
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (y_ptr[mid] <= t) lo = mid; else hi = mid;
    }
    y_of[t] = (int)lo;
    ent[t] = (int)t;
    const int x = x_idx[t];
    if (x < 0 || x >= n_x) {
        atomicExch(&status[G_ST_BAD], 1);
        return;
    }
    atomicAdd(&cnt[x], 1ull);
}

// occurrence index of every entry among those with the same (x, y): in the x-major order they are adjacent
__global__ void gen_occ_kernel(int64_t nnz, const int* __restrict__ x_ent, const int32_t* __restrict__ x_sorted,
                               const int* __restrict__ y_of, uint8_t* __restrict__ occ, int* status) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= nnz) return;
    const int e = x_ent[p];
    const int y = y_of[e];
    const int x = x_sorted[p];
    int k = 0;
    for (int64_t q = p - 1; q >= 0 && x_sorted[q] == x && y_of[x_ent[q]] == y; --q) ++k;
    if (k > 255) {
        atomicExch(&status[G_ST_BAD], 2);
        k = 255;
    }
    occ[e] = (uint8_t)k;
    if (k) atomicMax(&status[G_ST_MAXOCC], k);
}

// KIND: 0 cosine, 1 msd, 2 pearson, 3 pearson_baseline (SB2_SIM_*)
template <int KIND>
__global__ void __launch_bounds__(256) sim_rows_kernel(const GenArgs a) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int64_t n_x = a.n_x;
    // accumulators of the row, one record per column: a co-rating touches ONE 32-byte sector (two for pearson)
    constexpr int NREC = KIND == 2 ? 6 : 4;
    double* REC = a.scratch + (size_t)blockIdx.x * a.scratch_stride;
    constexpr int I_SQI = 1, I_SQJ = 2, I_SI = 3, I_SJ = 4, I_FQ = NREC - 1;  // [0] = prods (msd: sq_diff)
    int min_sprt = a.min_support;
    if (KIND == 3 && min_sprt < 2) min_sprt = 2;  // similarities.pyx:334
    for (int64_t ob = blockIdx.x; ob < a.n_rows; ob += gridDim.x) {
        const int64_t row = a.rows ? a.rows[ob] : a.row_begin + ob;
        for (int64_t x = tid; x < n_x * NREC; x += nthr) REC[x] = 0.0;   // freq is kept as a double (exact below 2^53)
        __syncthreads();
        const double bxi = KIND == 3 ? a.bx[row] : 0.0;
        // one co-rating (ri of this row's entry, rj of entry c): the reference's updates of acc[row, xj]; `up`: the
        // pair is evaluated as (xi = row, xj) -- otherwise as (xi = xj, xj = row), whose accumulators the finalize
        // reads for the lower triangle
        auto visit = [&](double ri, double di, double pb, int64_t c) {
            const int xj = a.x_idx[c];
            const double rj = a.r[c];
            double* R = REC + (size_t)xj * NREC;
            if (KIND == 2) {
                double2 v0 = *reinterpret_cast<double2*>(R), v1 = *reinterpret_cast<double2*>(R + 2),
                        v2 = *reinterpret_cast<double2*>(R + 4);
                v0.x = __dadd_rn(v0.x, __dmul_rn(ri, rj));
                v0.y = __dadd_rn(v0.y, __dmul_rn(ri, ri));
                v1.x = __dadd_rn(v1.x, __dmul_rn(rj, rj));
                v1.y = __dadd_rn(v1.y, ri);
                v2.x = __dadd_rn(v2.x, rj);
                v2.y += 1.0;
                *reinterpret_cast<double2*>(R) = v0; *reinterpret_cast<double2*>(R + 2) = v1;
                *reinterpret_cast<double2*>(R + 4) = v2;
            } else {
                double2 v0 = *reinterpret_cast<double2*>(R), v1 = *reinterpret_cast<double2*>(R + 2);
                if (KIND == 0) {
                    v0.x = __dadd_rn(v0.x, __dmul_rn(ri, rj));
                    v0.y = __dadd_rn(v0.y, __dmul_rn(ri, ri));
                    v1.x = __dadd_rn(v1.x, __dmul_rn(rj, rj));
                } else if (KIND == 1) {
                    const double d = __dsub_rn(ri, rj);
                    v0.x = __dadd_rn(v0.x, __dmul_rn(d, d));
                } else {
                    const double dj = __dsub_rn(rj, __dadd_rn(pb, a.bx[xj]));
                    v0.x = __dadd_rn(v0.x, __dmul_rn(di, dj));
                    v0.y = __dadd_rn(v0.y, __dmul_rn(di, di));
                    v1.x = __dadd_rn(v1.x, __dmul_rn(dj, dj));
                }
                v1.y += 1.0;
                *reinterpret_cast<double2*>(R) = v0; *reinterpret_cast<double2*>(R + 2) = v1;
            }
        };
        const int64_t p_end = a.x_ptr[row + 1];
        for (int64_t p = a.x_ptr[row]; p < p_end;) {
            const int64_t y = a.y_of[a.x_ent[p]];
            const int64_t b = a.y_ptr[y], e = a.y_ptr[y + 1];
            const double pb = KIND == 3 ? __dadd_rn(a.mu, a.by[y]) : 0.0;  // partial_bias, similarities.pyx:337
            if (a.max_occ == 0) {
                // no duplicated pair anywhere: one entry of this row per y, every column at most once per sweep
                const double ri = a.r[a.x_ent[p]];
                const double di = KIND == 3 ? __dsub_rn(ri, __dadd_rn(pb, bxi)) : 0.0;
                for (int64_t c = b + tid; c < e; c += nthr)
                    if (a.x_idx[c] >= a.col_begin) visit(ri, di, pb, c);
                __syncthreads();  // the next sweep may hit the same columns
                ++p;
                continue;
            }
            // duplicated pairs: the row has m >= 1 entries under this y (adjacent in the x-major order) and a column
            // may occur several times in yr[y].  The reference's order for the accumulators of the pair (xi, xj),
            // xi < xj, is: entries of xi outer, entries of xj inner.
            int64_t p1 = p + 1;
            while (p1 < p_end && a.y_of[a.x_ent[p1]] == y) ++p1;
            // columns >= row: this row is xi -> its entries outer, the column's copies in rounds of their occurrence
            for (int64_t q = p; q < p1; ++q) {
                const double ri = a.r[a.x_ent[q]];
                const double di = KIND == 3 ? __dsub_rn(ri, __dadd_rn(pb, bxi)) : 0.0;
                for (int round = 0; round <= a.max_occ; ++round) {
                    for (int64_t c = b + tid; c < e; c += nthr)
                        if (a.occ[c] == round && a.x_idx[c] >= row) visit(ri, di, pb, c);
                    __syncthreads();
                }
            }
            // columns < row: the column is xi -> its copies outer (rounds), this row's entries inner (one thread)
            for (int round = 0; round <= a.max_occ; ++round) {
                for (int64_t c = b + tid; c < e; c += nthr)
                    if (a.occ[c] == round && a.x_idx[c] < row && a.x_idx[c] >= a.col_begin)
                        for (int64_t q = p; q < p1; ++q) {
                            const double ri = a.r[a.x_ent[q]];
                            const double di = KIND == 3 ? __dsub_rn(ri, __dadd_rn(pb, bxi)) : 0.0;
                            visit(ri, di, pb, c);
                        }
                __syncthreads();
            }
            p = p1;
        }
        // finalize (similarities.pyx:86-95 / :155-164 / :240-256 / :347-359).  The reference evaluates pairs xi < xj
        // from the accumulators at [xi, xj] and mirrors; by symmetry of the definitions (sqi[xj, xi] == sqj[xi, xj]
        // etc., same terms in the same order) evaluating [row, xj] with the roles swapped for xj < row gives the
        // same bits (with duplicated pairs too: the accumulation above keeps the reference's loop nesting for the
        // columns below the diagonal), so every row is finished by its own CTA.
        double* out = a.sim + (size_t)ob * (size_t)a.out_ld;
        for (int64_t xj = a.col_begin + tid; xj < n_x; xj += nthr) {
            double s = 0.0;
            const double* R = REC + (size_t)xj * NREC;
            const int fq = (int)R[I_FQ];
            if (xj == row) {
                s = 1.0;
            } else if (fq >= min_sprt) {
                const bool up = row < xj;
                const double prods = R[0], sqi = up ? R[I_SQI] : R[I_SQJ], sqj = up ? R[I_SQJ] : R[I_SQI];
                if (KIND == 0) {
                    s = __ddiv_rn(prods, __dsqrt_rn(__dmul_rn(sqi, sqj)));
                } else if (KIND == 1) {
                    if (fq == 0) atomicExch(&a.status[G_ST_ZERODIV], 1);
                    else s = __ddiv_rn(1.0, __dadd_rn(__ddiv_rn(prods, (double)fq), 1.0));
                } else if (KIND == 2) {
                    const double n = (double)fq;
                    const double si = up ? R[I_SI] : R[I_SJ], sj = up ? R[I_SJ] : R[I_SI];
                    const double num = __dsub_rn(__dmul_rn(n, prods), __dmul_rn(si, sj));
                    const double denum = __dsqrt_rn(__dmul_rn(__dsub_rn(__dmul_rn(n, sqi), __dmul_rn(si, si)),
                                                              __dsub_rn(__dmul_rn(n, sqj), __dmul_rn(sj, sj))));
                    s = denum == 0.0 ? 0.0 : __ddiv_rn(num, denum);
                } else {
                    s = __ddiv_rn(prods, __dsqrt_rn(__dmul_rn(sqi, sqj)));
                    const double fm1 = (double)(fq - 1);
                    const double den = __dadd_rn(fm1, a.shrinkage);
                    if (den == 0.0) atomicExch(&a.status[G_ST_ZERODIV], 1);
                    else s = __dmul_rn(s, __ddiv_rn(fm1, den));
                }
            }
            out[xj] = s;
        }
        __syncthreads();
    }
}

// x-major sweep descriptors: one coalesced stream per row instead of the dependent chain
// x_ent -> y_of -> y_ptr -> entries in front of every sweep
__global__ void gen_desc_kernel(int64_t nnz, const int* __restrict__ x_ent, const int* __restrict__ y_of,
                                const int64_t* __restrict__ y_ptr, const double* __restrict__ val,
                                int64_t* __restrict__ xm_b, int* __restrict__ xm_len, double* __restrict__ xm_r) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= nnz) return;
    const int e = x_ent[p];
    const int y = y_of[e];
    const int64_t b = y_ptr[y];
    xm_b[p] = b;
    xm_len[p] = (int)(y_ptr[y + 1] - b);
    xm_r[p] = val[e];
}

// pearson_baseline: deviation of every entry, r - ((mu + b_y) + b_x), the reference's operations in the reference's
// order (similarities.pyx:337-340); it depends on the entry alone
__global__ void gen_dev_kernel(int64_t nnz, const int32_t* __restrict__ x_idx, const int* __restrict__ y_of,
                               const double* __restrict__ r, double mu, const double* __restrict__ bx,
                               const double* __restrict__ by, double* __restrict__ dev) {
    const int64_t c = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (c >= nnz) return;
    const double pb = __dadd_rn(mu, by[y_of[c]]);
    dev[c] = __dsub_rn(r[c], __dadd_rn(pb, bx[x_idx[c]]));
}

// The same accumulation as sim_rows_kernel for inputs WITHOUT duplicated pairs (one entry of the row per y, every
// column at most once per sweep), with the memory latencies taken off the critical path of a sweep:
//   * the sweep descriptors of a row (segment start / length, the row's value) arrive in coalesced chunks through
//     shared memory instead of the dependent chain x_ent -> y_of -> y_ptr in front of every sweep;
//   * the (x, value) entries of the sweeps stream through a shared-memory ring filled by cp.async, GEN_RING sweeps
//     ahead;
//   * pearson_baseline: the deviations r - ((mu + b_y) + b_x) depend on the ENTRY only, so they are computed once per
//     entry (gen_dev_kernel, the reference's operation order) and the accumulation becomes cosine's on deviations
//     -- no gather of b_x inside the sweeps.
// What remains per co-rating is the read-modify-write of one 32-byte column record (48 B for pearson) in the CTA's
// scratch row: ~1.3 TB/s of random 32-byte-sector DRAM traffic at the ml-20M shape (ncu: DRAM bytes ~= 64 B per
// co-rating, L2 hit rate 55 %), which is what bounds the kernel.  Keeping the records of a column TILE in shared
// memory instead (one CTA per SM, every tile re-reading the row's segments) was measured slower: 0.20 s against 0.14 s
// for cosine at that shape -- with one resident CTA per SM the per-sweep barrier and shared-memory latencies are not
// hidden (DESIGN.md section 10).
constexpr int GEN_CHUNK = 128;
constexpr int GEN_RING = 8;   // sweeps in flight
template <int KIND>
__global__ void __launch_bounds__(256, 4) sim_rows_fast_kernel(const GenArgs a) {
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int64_t n_x = a.n_x;
    constexpr int NREC = KIND == 2 ? 6 : 4;
    constexpr int I_SQI = 1, I_SQJ = 2, I_SI = 3, I_SJ = 4, I_FQ = NREC - 1;
    __shared__ int64_t s_b[GEN_CHUNK];
    __shared__ int s_len[GEN_CHUNK];
    __shared__ double s_r[GEN_CHUNK];
    __shared__ int s_x[GEN_RING][256];
    __shared__ double s_rj[GEN_RING][256];
    int min_sprt = a.min_support;
    if (KIND == 3 && min_sprt < 2) min_sprt = 2;  // similarities.pyx:334
    double* REC = a.scratch + (size_t)blockIdx.x * a.scratch_stride;   // this CTA's row of column records
    const int c0 = (int)a.col_begin, c1 = (int)n_x;
    for (int64_t ob = blockIdx.x; ob < a.n_rows; ob += gridDim.x) {
        const int64_t row = a.rows ? a.rows[ob] : a.row_begin + ob;
        for (int64_t x = tid; x < (int64_t)(c1 - c0) * NREC / 2; x += nthr)
            reinterpret_cast<double2*>(REC)[x] = make_double2(0.0, 0.0);
        // ri / rj: ratings -- or, for pearson_baseline, the precomputed deviations
        auto visit = [&](double ri, int xj, double rj) {
            double* R = REC + (size_t)(xj - c0) * NREC;
            if (KIND == 2) {
                double2 v0 = *reinterpret_cast<double2*>(R), v1 = *reinterpret_cast<double2*>(R + 2),
                        v2 = *reinterpret_cast<double2*>(R + 4);
                v0.x = __dadd_rn(v0.x, __dmul_rn(ri, rj));
                v0.y = __dadd_rn(v0.y, __dmul_rn(ri, ri));
                v1.x = __dadd_rn(v1.x, __dmul_rn(rj, rj));
                v1.y = __dadd_rn(v1.y, ri);
                v2.x = __dadd_rn(v2.x, rj);
                v2.y += 1.0;
                *reinterpret_cast<double2*>(R) = v0; *reinterpret_cast<double2*>(R + 2) = v1;
                *reinterpret_cast<double2*>(R + 4) = v2;
            } else {
                double2 v0 = *reinterpret_cast<double2*>(R), v1 = *reinterpret_cast<double2*>(R + 2);
                if (KIND == 1) {
                    const double d = __dsub_rn(ri, rj);
                    v0.x = __dadd_rn(v0.x, __dmul_rn(d, d));
                } else {
                    v0.x = __dadd_rn(v0.x, __dmul_rn(ri, rj));
                    v0.y = __dadd_rn(v0.y, __dmul_rn(ri, ri));
                    v1.x = __dadd_rn(v1.x, __dmul_rn(rj, rj));
                }
                v1.y += 1.0;
                *reinterpret_cast<double2*>(R) = v0; *reinterpret_cast<double2*>(R + 2) = v1;
            }
        };
        const int64_t p_end = a.x_ptr[row + 1];
        for (int64_t p0 = a.x_ptr[row]; p0 < p_end; p0 += GEN_CHUNK) {
            const int nq = (int)(p_end - p0 < GEN_CHUNK ? p_end - p0 : GEN_CHUNK);
            __syncthreads();   // the previous chunk's descriptors are no longer read; (first chunk) REC is zeroed
            if (tid < nq) {
                s_b[tid] = a.xm_b[p0 + tid]; s_len[tid] = a.xm_len[p0 + tid]; s_r[tid] = a.xm_r[p0 + tid];
            }
            __syncthreads();
            // (x, r) of the sweeps stream through a ring of GEN_RING stages filled by cp.async: the entries of sweep
            // q + GEN_RING - 1 are requested while sweep q is applied, so that the L2 latency (~4 sweeps long) is
            // hidden with one CTA per SM.  Every thread copies and later reads its OWN slot: no barrier is needed
            // between the copy and the read, only cp.async.wait_group.
            auto request = [&](int q) {
                if (q < nq && tid < s_len[q]) {
                    const int st = q % GEN_RING;
                    const int64_t c = s_b[q] + tid;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_x[st][tid])),
                                 "l"(a.x_idx + c) : "memory");
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(&s_rj[st][tid])),
                                 "l"(a.val + c) : "memory");
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            for (int q = 0; q < GEN_RING - 1; ++q) request(q);
            for (int q = 0; q < nq; ++q) {
                request(q + GEN_RING - 1);
                asm volatile("cp.async.wait_group %0;" ::"n"(GEN_RING - 1) : "memory");   // sweep q has landed
                const double ri = s_r[q];
                if (tid < s_len[q]) {
                    const int xj = s_x[q % GEN_RING][tid];
                    if (xj >= c0) visit(ri, xj, s_rj[q % GEN_RING][tid]);
                }
                for (int64_t c = s_b[q] + tid + nthr; c < s_b[q] + s_len[q]; c += nthr) {   // segments longer than the CTA
                    const int xc = a.x_idx[c];
                    if (xc >= c0) visit(ri, xc, a.val[c]);
                }
                __syncthreads();  // the next sweep may hit the same columns
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        // finalize (similarities.pyx:86-95 / :155-164 / :240-256 / :347-359); see sim_rows_kernel for why every row
        // can evaluate both triangles itself
        double* out = a.sim + (size_t)ob * (size_t)a.out_ld;
        for (int xj = c0 + tid; xj < c1; xj += nthr) {
            double s = 0.0;
            const double* R = REC + (size_t)(xj - c0) * NREC;
            const int fq = (int)R[I_FQ];
            if (xj == row) {
                s = 1.0;
            } else if (fq >= min_sprt) {
                const bool up = row < xj;
                const double prods = R[0], sqi = up ? R[I_SQI] : R[I_SQJ], sqj = up ? R[I_SQJ] : R[I_SQI];
                if (KIND == 0) {
                    s = __ddiv_rn(prods, __dsqrt_rn(__dmul_rn(sqi, sqj)));
                } else if (KIND == 1) {
                    if (fq == 0) atomicExch(&a.status[G_ST_ZERODIV], 1);
                    else s = __ddiv_rn(1.0, __dadd_rn(__ddiv_rn(prods, (double)fq), 1.0));
                } else if (KIND == 2) {
                    const double n = (double)fq;
                    const double si = up ? R[I_SI] : R[I_SJ], sj = up ? R[I_SJ] : R[I_SI];
                    const double num = __dsub_rn(__dmul_rn(n, prods), __dmul_rn(si, sj));
                    const double denum = __dsqrt_rn(__dmul_rn(__dsub_rn(__dmul_rn(n, sqi), __dmul_rn(si, si)),
                                                              __dsub_rn(__dmul_rn(n, sqj), __dmul_rn(sj, sj))));
                    s = denum == 0.0 ? 0.0 : __ddiv_rn(num, denum);
                } else {
                    s = __ddiv_rn(prods, __dsqrt_rn(__dmul_rn(sqi, sqj)));
                    const double fm1 = (double)(fq - 1);
                    const double den = __dadd_rn(fm1, a.shrinkage);
                    if (den == 0.0) atomicExch(&a.status[G_ST_ZERODIV], 1);
                    else s = __dmul_rn(s, __ddiv_rn(fm1, den));
                }
            }
            out[xj] = s;
        }
        __syncthreads();   // REC is zeroed for the next row only after every thread has read it
    }
}

// rows == nullptr: output rows are the matrix rows [row_begin, row_end).  Otherwise row_begin = 0 and output row b is
// matrix row rows[b] (b < row_end, the rows already checked to lie in [0, n_x)).  Output row b starts at sim_out + b * out_ld.
int sim_general_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                    int64_t nnz, int min_support, double global_mean, const double* x_biases, const double* y_biases,
                    double shrinkage, int64_t row_begin, int64_t row_end, const int32_t* rows, bool upper,
                    double* sim_out, int64_t out_ld, cudaStream_t st) {
    if (kind < 0 || kind > 3 || n_x <= 0 || n_y < 0 || nnz < 0 || nnz > 0x7FFFFFF0ll || row_begin < 0 ||
        (!rows && row_end > n_x) || (rows && (row_begin != 0 || upper)) || row_begin >= row_end || out_ld < n_x) {
        set_error("sim_build (general path): invalid argument");
        return SB2_ERR_INVALID;
    }
    if (kind == SB2_SIM_PEARSON_BASELINE && (!x_biases || !y_biases)) {
        set_error("sim_build: pearson_baseline needs x_biases and y_biases");
        return SB2_ERR_INVALID;
    }
    const size_t n1 = (size_t)std::max<int64_t>(nnz, 1);
    DevBuf status_d, y_of_d, ent_d, ent2_d, key2_d, cnt_d, xptr_d, occ_d, tmp_d, scratch_d;
    SB2_TRY(status_d.alloc(G_ST_NWORDS * sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(status_d.p, 0, G_ST_NWORDS * sizeof(int), st));
    SB2_TRY(y_of_d.alloc(n1 * 4, st));
    SB2_TRY(ent_d.alloc(n1 * 4, st));
    SB2_TRY(ent2_d.alloc(n1 * 4, st));
    SB2_TRY(key2_d.alloc(n1 * 4, st));
    SB2_TRY(occ_d.alloc(n1, st));
    SB2_TRY(cnt_d.alloc((size_t)(n_x + 1) * 8, st));
    SB2_TRY(xptr_d.alloc((size_t)(n_x + 1) * 8, st));
    SB2_CUDA(cudaMemsetAsync(cnt_d.p, 0, (size_t)(n_x + 1) * 8, st));
    SB2_CUDA(cudaMemsetAsync(occ_d.p, 0, n1, st));
    int bits = 1;
    while (((int64_t)1 << bits) < n_x) ++bits;
    size_t t1 = 0, t2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, x_idx, key2_d.as<int32_t>(), ent_d.as<int>(), ent2_d.as<int>(), (int)nnz, 0, bits, st);
    cub::DeviceScan::ExclusiveSum(nullptr, t2, cnt_d.as<int64_t>(), xptr_d.as<int64_t>(), (int)(n_x + 1), st);
    const size_t tb = std::max(t1, t2);
    SB2_TRY(tmp_d.alloc(tb + 16, st));
    if (nnz > 0) {
        const unsigned nb = (unsigned)ceil_div(nnz, 256);
        gen_entry_kernel<<<nb, 256, 0, st>>>(nnz, n_x, n_y, y_ptr, x_idx, y_of_d.as<int>(), ent_d.as<int>(),
                                             cnt_d.as<unsigned long long>(), status_d.as<int>());
        SB2_LAUNCH_CHECK();
        size_t tt = tb;
        SB2_CUDA(cub::DeviceRadixSort::SortPairs(tmp_d.p, tt, x_idx, key2_d.as<int32_t>(), ent_d.as<int>(), ent2_d.as<int>(),
                                                 (int)nnz, 0, bits, st));
        launch_counter()++;
        gen_occ_kernel<<<nb, 256, 0, st>>>(nnz, ent2_d.as<int>(), key2_d.as<int32_t>(), y_of_d.as<int>(), occ_d.as<uint8_t>(),
                                           status_d.as<int>());
        SB2_LAUNCH_CHECK();
    }
    size_t tt2 = tb;
    SB2_CUDA(cub::DeviceScan::ExclusiveSum(tmp_d.p, tt2, cnt_d.as<int64_t>(), xptr_d.as<int64_t>(), (int)(n_x + 1), st));
    launch_counter()++;
    int status_h[G_ST_NWORDS];
    SB2_CUDA(cudaMemcpyAsync(status_h, status_d.p, sizeof(status_h), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (status_h[G_ST_BAD] == 1) {
        set_error("sim_build: x index out of range");
        return SB2_ERR_INVALID;
    }
    if (status_h[G_ST_BAD] == 2) {
        set_error("sim_build: more than 255 copies of one (x, y) pair");
        return SB2_ERR_UNSUPPORTED;
    }
    const int64_t rows_n = row_end - row_begin;
    int per_sm = 4;
    if (const char* e = getenv("SB2_SIM_GENERAL_CTAS")) per_sm = std::max(1, std::min(8, atoi(e)));
    const int grid = (int)std::min<int64_t>(rows_n, (int64_t)sm_count() * per_sm);
    const int64_t stride = (6 * n_x + 7) & ~(int64_t)3;  // records of 4 doubles (6 for pearson) per column, 32 B aligned
    SB2_TRY(scratch_d.alloc((size_t)grid * (size_t)stride * sizeof(double), st));
    GenArgs a;
    memset(&a, 0, sizeof(a));
    a.n_x = n_x; a.n_y = n_y; a.nnz = nnz; a.y_ptr = y_ptr; a.x_idx = x_idx; a.r = r;
    a.x_ptr = xptr_d.as<int64_t>(); a.x_ent = ent2_d.as<int>(); a.y_of = y_of_d.as<int>(); a.occ = occ_d.as<uint8_t>();
    a.max_occ = status_h[G_ST_MAXOCC]; a.min_support = min_support; a.mu = global_mean; a.shrinkage = shrinkage;
    a.bx = x_biases; a.by = y_biases; a.row_begin = row_begin; a.n_rows = rows_n; a.rows = rows; a.sim = sim_out;
    a.out_ld = out_ld;
    a.col_begin = upper ? row_begin : 0;
    a.scratch = scratch_d.as<double>(); a.scratch_stride = stride; a.status = status_d.as<int>();
    DevBuf xmb_d, xml_d, xmr_d, xmp_d;
    if (a.max_occ == 0 && nnz > 0) {
        // no duplicated pair (the usual case): x-major sweep descriptors + the software-pipelined kernel
        SB2_TRY(xmb_d.alloc(n1 * 8, st));
        SB2_TRY(xml_d.alloc(n1 * 4, st));
        SB2_TRY(xmr_d.alloc(n1 * 8, st));
        const double* val = r;
        if (kind == SB2_SIM_PEARSON_BASELINE) {
            SB2_TRY(xmp_d.alloc(n1 * 8, st));
            gen_dev_kernel<<<(unsigned)ceil_div(nnz, 256), 256, 0, st>>>(nnz, x_idx, y_of_d.as<int>(), r, global_mean, x_biases,
                                                                        y_biases, xmp_d.as<double>());
            SB2_LAUNCH_CHECK();
            val = xmp_d.as<double>();
        }
        gen_desc_kernel<<<(unsigned)ceil_div(nnz, 256), 256, 0, st>>>(nnz, ent2_d.as<int>(), y_of_d.as<int>(), y_ptr, val,
                                                                     xmb_d.as<int64_t>(), xml_d.as<int>(), xmr_d.as<double>());
        SB2_LAUNCH_CHECK();
        a.xm_b = xmb_d.as<int64_t>(); a.xm_len = xml_d.as<int>(); a.xm_r = xmr_d.as<double>(); a.val = val;
        switch (kind) {
            case 0: sim_rows_fast_kernel<0><<<grid, 256, 0, st>>>(a); break;
            case 1: sim_rows_fast_kernel<1><<<grid, 256, 0, st>>>(a); break;
            case 2: sim_rows_fast_kernel<2><<<grid, 256, 0, st>>>(a); break;
            default: sim_rows_fast_kernel<3><<<grid, 256, 0, st>>>(a); break;
        }
    } else {
        switch (kind) {
            case 0: sim_rows_kernel<0><<<grid, 256, 0, st>>>(a); break;
            case 1: sim_rows_kernel<1><<<grid, 256, 0, st>>>(a); break;
            case 2: sim_rows_kernel<2><<<grid, 256, 0, st>>>(a); break;
            default: sim_rows_kernel<3><<<grid, 256, 0, st>>>(a); break;
        }
    }
    SB2_LAUNCH_CHECK();
    SB2_CUDA(cudaMemcpyAsync(status_h, status_d.p, sizeof(status_h), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (status_h[G_ST_ZERODIV]) {
        set_error("float division");
        return SB2_ERR_ZERO_DIVISION;
    }
    return SB2_OK;
}

}  // namespace sb2
