// Similarity matrices on the int8 tensor cores.
//
// Replaces similarities.pyx:28-361 of the reference.  The reference's triple loop
//     for y: for (xi, ri) in yr[y]: for (xj, rj) in yr[y]:  freq[xi,xj] += 1; prods[xi,xj] += ri*rj; ...
// is a set of masked dense contractions over y of the n_x x n_y rating matrix:
//     freq = M M^T   prods = R R^T   sqi = (R.R) M^T   sqj = M (R.R)^T   si = R M^T   sj = M R^T
// (M = [R != 0]).  Ratings are exact multiples of 1/denom, so q = r*denom is an integer; q, q^2 are
// split into base-256 digits, each digit panel is a u8 matrix, every digit-pair product runs on
// tcgen05.mma kind::i8 with exact int32 accumulation (sim_gemm.cu) and the digits are recombined in
// fp64 planes (exact below 2^53).  pearson_baseline's residuals r - (mu + b_y) - b_x are expanded
// algebraically so that the only non-integer operand is a per-y scalar a_y = mu + b_y, which is
// quantised to 47-bit fixed point and digit-split the same way; the b_x terms are applied in the fp64
// finalize kernel.  See DESIGN.md "Similarity path" for the algebra and the error bound.
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.cuh"
#include "sim_gemm.cuh"

namespace sb2 {

// status words written by the kernels (device int[8])
enum { ST_BAD_RATING = 0, ST_MAX_Q = 1, ST_DUP = 2, ST_ZERODIV = 3, ST_BAD_ROW = 4, ST_NWORDS = 8 };

__device__ __forceinline__ int64_t find_segment(const int64_t* __restrict__ ptr, int64_t n_seg, int64_t a) {
    int64_t lo = 0, hi = n_seg;  // largest s with ptr[s] <= a
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (ptr[mid] <= a) lo = mid; else hi = mid;
    }
    return lo;
}

// pass 1: check the ratings are integer multiples of 1/denom and find max q; a_y range for baselines
__global__ void sim_analyze_kernel(const double* __restrict__ r, int64_t nnz, double denom, int truncate,
                                   int* __restrict__ status,
                                   const double* __restrict__ y_biases, int64_t n_y, double global_mean,
                                   double* __restrict__ a_y, unsigned long long* __restrict__ a_minmax) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < nnz) {
        const double q = r[t] * denom;
        const double qr = truncate ? trunc(q) : rint(q);  // SlopeOne reads ratings into C ints (slope_one.pyx:52)
        if ((!truncate && !(fabs(q - qr) <= 1e-9 * fmax(1.0, fabs(q)))) || !(qr >= 0.0) || qr > 65535.0)
            atomicExch(&status[ST_BAD_RATING], 1);
        else
            atomicMax(&status[ST_MAX_Q], (int)qr);
    }
    if (y_biases != nullptr && t < n_y) {
        const double a = global_mean + y_biases[t];  // partial_bias, similarities.pyx:337
        a_y[t] = a;
        // order-preserving map double -> uint64 for atomicMin/Max
        unsigned long long b = (unsigned long long)__double_as_longlong(a);
        b = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
        atomicMin(&a_minmax[0], b);
        atomicMax(&a_minmax[1], b);
    }
}

struct PackArgs {
    const int64_t* y_ptr;
    const int32_t* x_idx;
    const double* r;
    int64_t nnz, n_y, k_pad;
    double denom;
    uint8_t* m_panel;
    uint8_t* q_panel[2];
    int nq;
    uint8_t* s_panel[4];
    int ns;
    // pearson_baseline only
    const double* a_y;
    double a_shift;  // integer shift c: a' = a - c >= 0
    double a_scale;  // 2^FB
    uint8_t* a_panel[6];
    uint8_t* c_panel[6];
    int na, nc;
    int* status;
    int64_t n_x;
    int64_t x_min;  // rows below x_min are not read by this build (shard of a symmetric multi-rank build): not packed
    int truncate;
};

// pass 2: scatter the yr CSR into the dense K-major u8 panels
__global__ void sim_pack_kernel(const PackArgs p) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= p.nnz) return;
    const int64_t y = find_segment(p.y_ptr, p.n_y, t);
    const int64_t x = p.x_idx[t];
    if (x < 0 || x >= p.n_x) {
        atomicExch(&p.status[ST_BAD_RATING], 2);
        return;
    }
    if (x < p.x_min) return;
    const size_t o = (size_t)x * (size_t)p.k_pad + (size_t)y;
    // mask byte through a word atomic so that a second (x, y) hit is detected
    unsigned* mw = reinterpret_cast<unsigned*>(p.m_panel + (o & ~(size_t)3));
    const unsigned sh = (unsigned)(o & 3) * 8;
    const unsigned old = atomicAdd(mw, 1u << sh);
    if ((old >> sh) & 0xFF) {
        atomicExch(&p.status[ST_DUP], 1);
        return;
    }
    const unsigned q = (unsigned)(p.truncate ? trunc(p.r[t]) : rint(p.r[t] * p.denom));
    for (int d = 0; d < p.nq; ++d) p.q_panel[d][o] = (uint8_t)((q >> (8 * d)) & 0xFF);
    const unsigned long long s = (unsigned long long)q * q;
    for (int d = 0; d < p.ns; ++d) p.s_panel[d][o] = (uint8_t)((s >> (8 * d)) & 0xFF);
    if (p.na) {
        const double ap = p.a_y[y] - p.a_shift;
        const unsigned long long af = (unsigned long long)rint(ap * p.a_scale);  // < 2^48
        for (int d = 0; d < p.na; ++d) p.a_panel[d][o] = (uint8_t)((af >> (8 * d)) & 0xFF);
        // af^2 < 2^96: keep bits [48, 96)
        const unsigned long long hi = __umul64hi(af, af), lo = af * af;
        const unsigned long long cf = (hi << 16) | (lo >> 48);
        for (int d = 0; d < p.nc; ++d) p.c_panel[d][o] = (uint8_t)((cf >> (8 * d)) & 0xFF);
    }
}

// ----------------------------------------------------------------------------------------------
// finalize: planes -> sim.  All arithmetic in round-to-nearest fp64 with the reference's operation
// order and no FMA contraction (similarities.pyx:86-95, :155-164, :240-256, :347-359).
// ----------------------------------------------------------------------------------------------
struct FinArgs {
    int kind;
    int64_t n_x, ld;           // planes: rows x ld
    int64_t row_begin, row_end;  // global rows covered by this build (output rows are relative to row_begin)
    int64_t band_begin, band_end;  // rows finalized by this launch (their planes are resident)
    int64_t plane_row0;          // global row of plane row 0
    const double* freq;
    const double* prods;
    const double* sqi;
    const double* sqj;
    const double* si;
    const double* sj;
    const double* t1ij;
    const double* t1ji;
    const double* t2;
    const double* a1;
    const double* bx;
    double a_shift;
    double inv_d, inv_d2;  // 1/denom, 1/denom^2
    int min_support;
    double shrinkage;
    double* sim;  // (row_end-row_begin) x n_x; rows kernel: output row b at sim + (b - row_begin) * out_ld
    int64_t out_ld;
    const int32_t* rows;  // row list of sb2_sim_build_rows_dev: output (and plane) row b is matrix row rows[b]
    int* status;
};

// value of sim at (lo, hi) given the accumulators seen from (i, j); swap = (i > j)
__device__ __forceinline__ double sim_value(const FinArgs& f, size_t o, int64_t i, int64_t j, bool swap) {
    const double n = f.freq[o];
    if (n < (double)f.min_support) return 0.0;
    const double prods = __dmul_rn(f.prods[o], f.inv_d2);
    if (f.kind == SB2_SIM_MSD) {
        const double sqi = __dmul_rn(f.sqi[o], f.inv_d2), sqj = __dmul_rn(f.sqj[o], f.inv_d2);
        // sum (ri-rj)^2 = sqi + sqj - 2 prods: every term is an exact multiple of 1/denom^2
        const double sq_diff = __dsub_rn(__dadd_rn(sqi, sqj), __dmul_rn(2.0, prods));
        if (n == 0.0) {
            atomicExch(&f.status[ST_ZERODIV], 1);
            return 0.0;
        }
        return __ddiv_rn(1.0, __dadd_rn(__ddiv_rn(sq_diff, n), 1.0));
    }
    double sqi = __dmul_rn((swap ? f.sqj : f.sqi)[o], f.inv_d2);
    double sqj = __dmul_rn((swap ? f.sqi : f.sqj)[o], f.inv_d2);
    if (f.kind == SB2_SIM_COSINE) {
        const double denum = __dsqrt_rn(__dmul_rn(sqi, sqj));
        return __ddiv_rn(prods, denum);
    }
    const double si = __dmul_rn((swap ? f.sj : f.si)[o], f.inv_d);
    const double sj = __dmul_rn((swap ? f.si : f.sj)[o], f.inv_d);
    if (f.kind == SB2_SIM_PEARSON) {
        const double num = __dsub_rn(__dmul_rn(n, prods), __dmul_rn(si, sj));
        const double vi = __dsub_rn(__dmul_rn(n, sqi), __dmul_rn(si, si));
        const double vj = __dsub_rn(__dmul_rn(n, sqj), __dmul_rn(sj, sj));
        const double denum = __dsqrt_rn(__dmul_rn(vi, vj));
        return denum == 0.0 ? 0.0 : __ddiv_rn(num, denum);
    }
    // pearson_baseline: lo = min(i, j) plays "xi"
    const int64_t lo = swap ? j : i, hi = swap ? i : j;
    const double bi = f.bx[lo] + f.a_shift, bj = f.bx[hi] + f.a_shift;
    const double t1i = (swap ? f.t1ji : f.t1ij)[o], t1j = (swap ? f.t1ij : f.t1ji)[o];
    const double t2 = f.t2[o], a1 = f.a1[o];
    const double pr = prods - t1i - t1j + t2 - bj * si - bi * sj + (bi + bj) * a1 + bi * bj * n;
    double di = sqi - 2.0 * t1i + t2 - 2.0 * bi * si + 2.0 * bi * a1 + bi * bi * n;
    double dj = sqj - 2.0 * t1j + t2 - 2.0 * bj * sj + 2.0 * bj * a1 + bj * bj * n;
    di = fmax(di, 0.0);
    dj = fmax(dj, 0.0);
    double s = __ddiv_rn(pr, __dsqrt_rn(__dmul_rn(di, dj)));
    const double fm1 = n - 1.0;
    const double den = __dadd_rn(fm1, f.shrinkage);
    if (den == 0.0) {
        atomicExch(&f.status[ST_ZERODIV], 1);
        return 0.0;
    }
    s = __dmul_rn(s, __ddiv_rn(fm1, den));
    return s;
}

// symmetric build: 32x32 tiles with tj >= ti; the tile's values go to sim[i][j] and (transposed through shared
// memory) to sim[j][i], exactly like the reference mirrors (similarities.pyx:95).  Rows [f.band_begin, f.band_end)
// of the matrix are finalized per launch (their planes are resident); output rows are relative to f.row_begin
// (0 for the single-GPU build, the shard's first row for an upper-only shard), and the mirror is written only
// when the column is itself a row this build owns (j < f.row_end).
__global__ void sim_finalize_sym_kernel(const FinArgs f) {
    __shared__ double tile[32][33];
    const int ti = (int)(f.band_begin / 32) + blockIdx.y, tj = blockIdx.x;
    if (tj < ti) return;
    const int tx = threadIdx.x, ty0 = threadIdx.y;  // block 32 x 8
    for (int ty = ty0; ty < 32; ty += 8) {
        const int64_t i = (int64_t)ti * 32 + ty, j = (int64_t)tj * 32 + tx;
        double s = 0.0;
        if (i < f.band_end && j < f.n_x) {
            if (i == j) s = 1.0;
            else if (i < j) s = sim_value(f, (size_t)(i - f.plane_row0) * f.ld + j, i, j, false);
            if (i <= j) f.sim[(size_t)(i - f.row_begin) * f.n_x + j] = s;
        }
        tile[ty][tx] = s;
    }
    __syncthreads();
    for (int ty = ty0; ty < 32; ty += 8) {
        // element (row = tj*32+ty, col = ti*32+tx) = value at (col, row)
        const int64_t i = (int64_t)tj * 32 + ty, j = (int64_t)ti * 32 + tx;
        if (i < f.row_end && j < f.band_end && j < i) f.sim[(size_t)(i - f.row_begin) * f.n_x + j] = tile[tx][ty];
    }
}

// row-shard or row-list build: every (i, j) of the output rows, accumulators valid at (i, j) itself.  sim_value reads
// the accumulators of (i, j) with the roles swapped below the diagonal, which gives the bits the symmetric build
// mirrors from (j, i): every plane holds exact integer sums (or, for pearson_baseline, the same digit products in the
// same order on either side).
__global__ void sim_finalize_rows_kernel(const FinArgs f) {
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t b = f.band_begin + blockIdx.y;
    if (j >= f.n_x || b >= f.band_end) return;
    const int64_t i = f.rows ? f.rows[b] : b;
    double s;
    if (i == j) s = 1.0;
    else s = sim_value(f, (size_t)(b - f.plane_row0) * f.ld + j, i, j, i > j);
    f.sim[(size_t)(b - f.row_begin) * f.out_ld + j] = s;
}

// A-side panels of a row-list build: slot b of every panel is a copy of panel row rows[b]
__global__ void sim_gather_rows_kernel(const uint8_t* __restrict__ src, size_t src_panel_bytes, uint8_t* __restrict__ dst,
                                       size_t dst_panel_bytes, int n_panels, const int32_t* __restrict__ rows,
                                       int64_t n_rows, int64_t k_pad) {
    const int64_t per_row = k_pad / 16, per_panel = n_rows * per_row;
    for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < per_panel * n_panels;
         t += (int64_t)gridDim.x * blockDim.x) {
        const int64_t q = t / per_panel, rem = t - q * per_panel, b = rem / per_row, c = rem - b * per_row;
        const uint4* s = reinterpret_cast<const uint4*>(src + q * src_panel_bytes + (size_t)rows[b] * k_pad);
        reinterpret_cast<uint4*>(dst + q * dst_panel_bytes + (size_t)b * k_pad)[c] = s[c];
    }
}

__global__ void sim_check_rows_kernel(const int32_t* __restrict__ rows, int64_t n_rows, int64_t n_x, int* status) {
    const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (b < n_rows && (rows[b] < 0 || rows[b] >= n_x)) atomicExch(&status[ST_BAD_ROW], 1);
}

// SlopeOne (slope_one.pyx:59-70): freq[i][j] = |U_ij| (int64, symmetric, diagonal = raters of i);
// dev[i][j] = (sum_{u in U_ij} r_ui - r_uj) / freq[i][j] for i < j (0 / 0 = NaN where no common user),
// dev[j][i] = -dev[i][j], dev[i][i] = 0.  The sums are integers (ratings truncated to C ints), so
// si - sj below is the reference's accumulated value exactly.  Same 32x32 tile walk as the symmetric
// similarity finalize.
__global__ void slope_finalize_kernel(const FinArgs f, int64_t* __restrict__ freq_out, double* __restrict__ dev_out) {
    __shared__ double tdev[32][33];
    __shared__ double tfreq[32][33];
    const int ti = (int)(f.band_begin / 32) + blockIdx.y, tj = blockIdx.x;
    if (tj < ti) return;
    const int tx = threadIdx.x, ty0 = threadIdx.y;
    for (int ty = ty0; ty < 32; ty += 8) {
        const int64_t i = (int64_t)ti * 32 + ty, j = (int64_t)tj * 32 + tx;
        double d = 0.0, n = 0.0;
        if (i < f.band_end && j < f.n_x && i <= j) {
            const size_t o = (size_t)(i - f.plane_row0) * f.ld + j;
            n = f.freq[o];
            if (i < j) d = __ddiv_rn(__dsub_rn(f.si[o], f.sj[o]), n);
            freq_out[(size_t)i * f.n_x + j] = (int64_t)n;
            dev_out[(size_t)i * f.n_x + j] = d;
        }
        tdev[ty][tx] = d;
        tfreq[ty][tx] = n;
    }
    __syncthreads();
    for (int ty = ty0; ty < 32; ty += 8) {
        const int64_t i = (int64_t)tj * 32 + ty, j = (int64_t)ti * 32 + tx;
        if (i < f.n_x && j < f.band_end && j < i) {
            freq_out[(size_t)i * f.n_x + j] = (int64_t)tfreq[tx][ty];
            dev_out[(size_t)i * f.n_x + j] = -tdev[tx][ty];
        }
    }
}

// ----------------------------------------------------------------------------------------------
// driver
// ----------------------------------------------------------------------------------------------
static int n_digits(unsigned long long v) {
    int d = 1;
    while (v >>= 8) ++d;
    return d;
}

constexpr int KIND_SLOPE_ONE = 4;  // internal: freq + dev of SlopeOne from the FREQ / SI / SJ planes

// rows == nullptr: the matrix rows [row_begin, row_end).  Otherwise a row-list build: row_begin = 0, output row b
// (b < row_end) is matrix row rows[b] (checked to lie in [0, n_x)), written at sim_out + b * out_ld.  Its A-side panels
// hold the listed rows only (gathered from the full panels, which stay the B side), and the row blocks of the GEMM and
// the finalize walk the list's slots: 2 G n_rows n_x n_y operations, no symmetry.
static int sim_core(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                    int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                    const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end,
                    const int32_t* rows, double* sim_out, int64_t out_ld, int64_t* freq_out, bool upper,
                    cudaStream_t st) {
    const bool slope = (kind == KIND_SLOPE_ONE);
    if (kind < 0 || kind > 4 || n_x <= 0 || n_y < 0 || nnz < 0 || rating_denom <= 0 || row_begin < 0 ||
        (!rows && row_end > n_x) || (rows && (row_begin != 0 || upper || slope)) || row_begin >= row_end) {
        set_error("sim_build: invalid argument");
        return SB2_ERR_INVALID;
    }
    const bool pb = (kind == SB2_SIM_PEARSON_BASELINE);
    if (pb && (!x_biases || !y_biases)) {
        set_error("sim_build: pearson_baseline needs x_biases and y_biases");
        return SB2_ERR_INVALID;
    }
    if (pb && min_support < 2) min_support = 2;  // similarities.pyx:334
    const bool full = (!rows && row_begin == 0 && row_end == n_x);
    const int TR = gemm_tile_rows();  // 256 (CTA-pair kernel) or 128
    if (!full && row_begin % TR) {
        set_error("sim_build: row_begin of a shard must be a multiple of %d", TR);
        return SB2_ERR_INVALID;
    }
    const int64_t n_pad = round_up(n_x, TR);
    const int64_t k_pad = round_up(std::max<int64_t>(n_y, 1), GEMM_BK);  // 128
    const int64_t rows_pad = round_up(row_end, TR) - row_begin;  // plane rows (shard, or slots of a row list)
    const int64_t ld = n_pad;

    // ---- pass 1: analyse ratings --------------------------------------------------------------
    DevBuf status_d, a_y_d, mm_d;
    SB2_TRY(status_d.alloc(ST_NWORDS * sizeof(int), st));
    SB2_CUDA(cudaMemsetAsync(status_d.p, 0, ST_NWORDS * sizeof(int), st));
    SB2_TRY(mm_d.alloc(2 * sizeof(unsigned long long), st));
    const unsigned long long mm_init[2] = {~0ull, 0ull};
    SB2_CUDA(cudaMemcpyAsync(mm_d.p, mm_init, sizeof(mm_init), cudaMemcpyHostToDevice, st));
    if (pb) SB2_TRY(a_y_d.alloc((size_t)std::max<int64_t>(n_y, 1) * sizeof(double), st));
    {
        const int64_t work = std::max(nnz, pb ? n_y : (int64_t)0);
        if (work > 0) {
            sim_analyze_kernel<<<(unsigned)ceil_div(work, 256), 256, 0, st>>>(
                r, nnz, (double)rating_denom, slope ? 1 : 0, status_d.as<int>(), pb ? y_biases : nullptr, n_y, global_mean,
                a_y_d.as<double>(), mm_d.as<unsigned long long>());
            SB2_LAUNCH_CHECK();
        }
    }
    int status_h[ST_NWORDS];
    unsigned long long mm_h[2];
    SB2_CUDA(cudaMemcpyAsync(status_h, status_d.p, sizeof(status_h), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaMemcpyAsync(mm_h, mm_d.p, sizeof(mm_h), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (status_h[ST_BAD_RATING]) {
        if (slope) set_error("slope_one: ratings outside [0, 65535]");
        else set_error("sim_build: ratings are not integer multiples of 1/%d in [0, 65535/%d]", rating_denom,
                       rating_denom);
        return SB2_ERR_UNSUPPORTED;
    }
    const unsigned long long max_q = (unsigned long long)status_h[ST_MAX_Q];
    const int nq = n_digits(max_q), ns = slope ? 0 : n_digits(max_q * max_q);

    double a_shift = 0.0, a_scale = 1.0;
    int FB = 0, na = 0, nc = 0;
    if (pb) {
        auto unmap = [](unsigned long long b) {
            b = (b >> 63) ? (b & 0x7FFFFFFFFFFFFFFFull) : ~b;
            double d;
            memcpy(&d, &b, sizeof(d));
            return d;
        };
        double amin = n_y > 0 ? unmap(mm_h[0]) : 0.0, amax = n_y > 0 ? unmap(mm_h[1]) : 0.0;
        if (!(amin == amin) || !(amax == amax) || fabs(amin) > 1e12 || fabs(amax) > 1e12) {
            set_error("sim_build: non-finite baselines");
            return SB2_ERR_INVALID;
        }
        a_shift = floor(amin);
        const double range = amax - a_shift;  // a' in [0, range]
        int ib = 1;
        while (ldexp(1.0, ib) <= range) ++ib;
        FB = 47 - ib;  // a' * 2^FB < 2^47 (+ rounding) fits 6 base-256 digits
        if (FB < 16) {
            set_error("sim_build: baseline range too wide for the fixed-point path");
            return SB2_ERR_UNSUPPORTED;
        }
        a_scale = ldexp(1.0, FB);
        na = 6;
        nc = 6;
    }

    // ---- panels -------------------------------------------------------------------------------
    const size_t panel_bytes = (size_t)n_pad * (size_t)k_pad;
    const int n_panels = 1 + nq + ns + na + nc;
    DevBuf panels_d;
    SB2_TRY(panels_d.alloc(panel_bytes * n_panels, st));
    uint8_t* base = panels_d.as<uint8_t>();
    // a shard of a symmetric build (tiles at or above the block diagonal) reads panel rows >= row_begin only: the last
    // of 8 ranks clears and packs a quarter of the 56 GB of panels (ml-20M shape) instead of all of them
    const int64_t x_min = upper ? row_begin : 0;
    if (x_min == 0) {
        SB2_CUDA(cudaMemsetAsync(base, 0, panel_bytes * n_panels, st));
    } else {
        for (int q = 0; q < n_panels; ++q)
            SB2_CUDA(cudaMemsetAsync(base + panel_bytes * q + (size_t)x_min * (size_t)k_pad, 0,
                                     (size_t)(n_pad - x_min) * (size_t)k_pad, st));
    }
    int pi = 0;
    PackArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.y_ptr = y_ptr; pa.x_idx = x_idx; pa.r = r; pa.nnz = nnz; pa.n_y = n_y; pa.k_pad = k_pad;
    pa.denom = (double)rating_denom; pa.n_x = n_x; pa.x_min = x_min; pa.truncate = slope ? 1 : 0;
    pa.m_panel = base + panel_bytes * (pi++);
    pa.nq = nq; pa.ns = ns; pa.na = na; pa.nc = nc;
    for (int d = 0; d < nq; ++d) pa.q_panel[d] = base + panel_bytes * (pi++);
    for (int d = 0; d < ns; ++d) pa.s_panel[d] = base + panel_bytes * (pi++);
    for (int d = 0; d < na; ++d) pa.a_panel[d] = base + panel_bytes * (pi++);
    for (int d = 0; d < nc; ++d) pa.c_panel[d] = base + panel_bytes * (pi++);
    pa.a_y = a_y_d.as<double>(); pa.a_shift = a_shift; pa.a_scale = a_scale;
    pa.status = status_d.as<int>();
    if (nnz > 0) {
        sim_pack_kernel<<<(unsigned)ceil_div(nnz, 256), 256, 0, st>>>(pa);
        SB2_LAUNCH_CHECK();
    }
    DevBuf a_panels_d;
    const size_t a_panel_bytes = (size_t)rows_pad * (size_t)k_pad;
    if (rows) {
        SB2_TRY(a_panels_d.alloc(a_panel_bytes * n_panels, st));
        SB2_CUDA(cudaMemsetAsync(a_panels_d.p, 0, a_panel_bytes * n_panels, st));
        const int64_t n16 = row_end * (k_pad / 16) * n_panels;
        sim_gather_rows_kernel<<<(unsigned)std::min<int64_t>(ceil_div(n16, 256), 65536), 256, 0, st>>>(
            base, panel_bytes, a_panels_d.as<uint8_t>(), a_panel_bytes, n_panels, rows, row_end, k_pad);
        SB2_LAUNCH_CHECK();
    }

    // ---- planes + jobs ------------------------------------------------------------------------
    enum { P_FREQ, P_PRODS, P_SQI, P_SQJ, P_SI, P_SJ, P_T1IJ, P_T1JI, P_T2, P_A1, P_COUNT };
    bool need[P_COUNT] = {true, !slope, !slope, !slope, false, false, false, false, false, false};
    if (kind == SB2_SIM_PEARSON || pb || slope) need[P_SI] = need[P_SJ] = true;
    if (pb) need[P_T1IJ] = need[P_T1JI] = need[P_T2] = need[P_A1] = true;
    int n_planes = 0;
    int plane_slot[P_COUNT];
    for (int k = 0; k < P_COUNT; ++k) plane_slot[k] = need[k] ? n_planes++ : -1;
    // The fp64 planes cover one BAND of row blocks at a time (GEMMs, then finalize, band after band), so their
    // footprint is bounded (default 12 GiB; SB2_SIM_PLANE_GIB / SB2_SIM_BAND_ROWS override) instead of growing with
    // rows x n_x x 10: at the ml-20M item-item shape 59 GB of planes become 12 -- and the build gets faster, 1.04 ->
    // 0.92 s (budget 48 / 24 / 12 / 6 / 3 GiB: 1.02 / 0.94 / 0.92 / 0.96 / 0.99 s) -- and a 47k-row shard of a
    // 138k x 138k user-user build (52 GB of output) still fits one 180 GB GPU.
    const int rb0 = (int)(row_begin / TR), rb1 = (int)ceil_div(row_end, TR);
    int band_rb = rb1 - rb0;
    {
        double gib = 12.0;
        if (const char* e = getenv("SB2_SIM_PLANE_GIB")) gib = std::max(0.001, atof(e));
        const double per_rb = (double)n_planes * (double)ld * 8.0 * TR;
        band_rb = (int)std::max(1.0, std::min((double)band_rb, floor(gib * 1073741824.0 / per_rb)));
        if (const char* e = getenv("SB2_SIM_BAND_ROWS")) band_rb = std::max(1, std::min(rb1 - rb0, atoi(e) / TR));
        if (band_rb >= 8 && band_rb < rb1 - rb0) band_rb -= band_rb % 8;  // keep the 8-row-block L2 groups intact
    }
    const size_t plane_elems = (size_t)std::min<int64_t>(rows_pad, (int64_t)band_rb * TR) * (size_t)ld;
    DevBuf planes_d;
    SB2_TRY(planes_d.alloc(plane_elems * sizeof(double) * n_planes, st));
    auto plane = [&](int k) -> double* {
        return plane_slot[k] < 0 ? nullptr : planes_d.as<double>() + plane_elems * plane_slot[k];
    };

    std::vector<GemmJob> jobs;
    bool started[P_COUNT] = {false};
    auto add = [&](int pl, const uint8_t* a, const uint8_t* b, double alpha) {
        jobs.push_back(GemmJob{a, b, plane(pl), alpha, started[pl] ? 1 : 0});
        started[pl] = true;
    };
    const uint8_t* M = pa.m_panel;
    add(P_FREQ, M, M, 1.0);
    // most significant digit pair first (keeps partial sums exact and ordered by magnitude)
    for (int s = 2 * (nq - 1); s >= 0 && need[P_PRODS]; --s)
        for (int a = nq - 1; a >= 0; --a) {
            const int b = s - a;
            if (b < 0 || b >= nq) continue;
            add(P_PRODS, pa.q_panel[a], pa.q_panel[b], ldexp(1.0, 8 * s));
        }
    for (int d = ns - 1; d >= 0; --d) {
        add(P_SQI, pa.s_panel[d], M, ldexp(1.0, 8 * d));
        add(P_SQJ, M, pa.s_panel[d], ldexp(1.0, 8 * d));
    }
    if (need[P_SI])
        for (int d = nq - 1; d >= 0; --d) {
            add(P_SI, pa.q_panel[d], M, ldexp(1.0, 8 * d));
            add(P_SJ, M, pa.q_panel[d], ldexp(1.0, 8 * d));
        }
    if (pb) {
        const double inv_d = 1.0 / (double)rating_denom;
        for (int s = na - 1; s >= 0; --s) {
            for (int d = nq - 1; d >= 0; --d) {
                const double alpha = ldexp(1.0, 8 * (s + d) - FB) * inv_d;
                add(P_T1IJ, pa.q_panel[d], pa.a_panel[s], alpha);
                add(P_T1JI, pa.a_panel[s], pa.q_panel[d], alpha);
            }
            add(P_A1, M, pa.a_panel[s], ldexp(1.0, 8 * s - FB));
        }
        for (int s = nc - 1; s >= 0; --s) add(P_T2, M, pa.c_panel[s], ldexp(1.0, 8 * s + 48 - 2 * FB));
    }
    // Order the jobs so that the two accumulators of a launch share an operand panel on the same side where they can
    // (3 operand tiles per pipeline stage instead of 4: less TMA and shared-memory fill traffic per MMA).  Jobs of
    // one plane keep their relative order (the first one overwrites, the rest accumulate) and never share a launch.
    {
        std::vector<GemmJob> ordered;
        std::vector<char> used(jobs.size(), 0);
        auto first_of_plane = [&](size_t k) {  // no earlier unused job writes the same plane
            for (size_t e = 0; e < k; ++e)
                if (!used[e] && jobs[e].out == jobs[k].out) return false;
            return true;
        };
        for (size_t k = 0; k < jobs.size(); ++k) {
            if (used[k]) continue;
            used[k] = 1;
            ordered.push_back(jobs[k]);
            int best = -1, best_share = 0;
            for (size_t m = k + 1; m < jobs.size(); ++m) {
                if (used[m] || jobs[m].out == jobs[k].out || !first_of_plane(m)) continue;
                const int share = (jobs[m].a == jobs[k].a) + (jobs[m].b == jobs[k].b);
                if (share > best_share) { best_share = share; best = (int)m; }
            }
            if (best < 0)  // nothing shares: take the next eligible job so that launches stay full
                for (size_t m = k + 1; m < jobs.size() && best < 0; ++m)
                    if (!used[m] && jobs[m].out != jobs[k].out && first_of_plane(m)) best = (int)m;
            if (best >= 0) {
                used[best] = 1;
                ordered.push_back(jobs[best]);
            }
        }
        jobs.swap(ordered);
    }
    if (rows)  // the A side of every job reads the same panel's gathered rows
        for (GemmJob& jb : jobs)
            jb.a = a_panels_d.as<uint8_t>() + (size_t)(jb.a - base) / panel_bytes * a_panel_bytes;
    const bool timing = getenv("SB2_SIM_TIMING") != nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (timing) {
        cudaEventCreate(&ev0);
        cudaEventCreate(&ev1);
        cudaEventRecord(ev0, st);
    }
    // ---- tile list: all bands, one upload ------------------------------------------------------
    // Inside a band of planes, row blocks are walked in groups of 8 and tiles go column-block-major, so the ~148
    // tiles in flight share ~8 A-side and ~8 B-side row blocks of every panel (L2 reuse).
    std::vector<int2> tiles;
    std::vector<size_t> band_off;
    {
        const int ncb = (int)(n_pad / TR);
        const int grp = TR == 256 ? 8 : 12;
        for (int p0 = rb0; p0 < rb1; p0 += band_rb) {
            band_off.push_back(tiles.size());
            const int p1 = std::min(p0 + band_rb, rb1);
            for (int b0 = p0; b0 < p1; b0 += grp)
                for (int cb = 0; cb < ncb; ++cb)
                    for (int rb = b0; rb < std::min(b0 + grp, p1); ++rb)
                        if ((!full && !upper) || cb >= rb) tiles.push_back(make_int2(rb, cb));
        }
        band_off.push_back(tiles.size());
    }
    DevBuf tiles_d;
    SB2_TRY(tiles_d.alloc(tiles.size() * sizeof(int2) + 16, st));
    SB2_CUDA(cudaMemcpyAsync(tiles_d.p, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, st));

    FinArgs f;
    memset(&f, 0, sizeof(f));
    f.kind = kind; f.n_x = n_x; f.ld = ld; f.row_begin = row_begin; f.row_end = row_end;
    f.freq = plane(P_FREQ); f.prods = plane(P_PRODS); f.sqi = plane(P_SQI); f.sqj = plane(P_SQJ);
    f.si = plane(P_SI); f.sj = plane(P_SJ); f.t1ij = plane(P_T1IJ); f.t1ji = plane(P_T1JI);
    f.t2 = plane(P_T2); f.a1 = plane(P_A1);
    f.bx = x_biases; f.a_shift = a_shift;
    f.inv_d = 1.0 / (double)rating_denom;
    f.inv_d2 = 1.0 / ((double)rating_denom * (double)rating_denom);
    f.min_support = min_support; f.shrinkage = shrinkage; f.sim = sim_out; f.status = status_d.as<int>();
    f.out_ld = rows ? out_ld : n_x; f.rows = rows;
    const unsigned nt = (unsigned)ceil_div(n_x, 32);
    for (size_t bi = 0; bi + 1 < band_off.size(); ++bi) {
        const int64_t band_begin = ((int64_t)rb0 + (int64_t)bi * band_rb) * TR;
        const int64_t band_end = std::min<int64_t>(row_end, band_begin + (int64_t)band_rb * TR);
        const size_t t0 = band_off[bi], nt_band = band_off[bi + 1] - t0;
        if (nt_band)
            SB2_TRY(gemm_u8_tc_run2(jobs.data(), (int)jobs.size(), rows ? rows_pad : n_pad, n_pad, k_pad,
                                    tiles_d.as<int2>() + t0, (int)nt_band, ld, band_begin, st));
        f.band_begin = band_begin; f.band_end = band_end; f.plane_row0 = band_begin;
        const unsigned rows32 = (unsigned)ceil_div(band_end - band_begin, 32);
        if (slope) slope_finalize_kernel<<<dim3(nt, rows32), dim3(32, 8), 0, st>>>(f, freq_out, sim_out);
        else if (full || upper) sim_finalize_sym_kernel<<<dim3(nt, rows32), dim3(32, 8), 0, st>>>(f);
        else
            for (int64_t c0 = band_begin; c0 < band_end; c0 += 65535) {  // gridDim.y <= 65535
                f.band_begin = c0;
                f.band_end = std::min<int64_t>(band_end, c0 + 65535);
                sim_finalize_rows_kernel<<<dim3((unsigned)ceil_div(n_x, 256), (unsigned)(f.band_end - c0)), 256, 0, st>>>(f);
            }
        SB2_LAUNCH_CHECK();
    }
    if (timing) {
        cudaEventRecord(ev1, st);
        cudaEventSynchronize(ev1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev0, ev1);
        const double ops = 2.0 * (double)jobs.size() * (double)tiles.size() * TR * TR * (double)k_pad;
        fprintf(stderr, "[sb2] sim gemm + finalize: %d accumulators x %zu tiles x k=%lld in %d band(s): %.3f ms, %.1f TOP/s issued\n",
                (int)jobs.size(), tiles.size(), (long long)k_pad, (int)ceil_div(rb1 - rb0, band_rb), ms,
                ops / (ms * 1e-3) / 1e12);
        cudaEventDestroy(ev0);
        cudaEventDestroy(ev1);
    }

    SB2_CUDA(cudaMemcpyAsync(status_h, status_d.p, sizeof(status_h), cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (status_h[ST_BAD_RATING]) {
        set_error("sim_build: x index out of range");
        return SB2_ERR_INVALID;
    }
    if (status_h[ST_DUP]) {
        set_error("sim_build: duplicate (x, y) pair in yr -- not representable in the dense rating panels");
        return SB2_ERR_DUPLICATE;
    }
    if (status_h[ST_ZERODIV]) {
        set_error("float division");
        return SB2_ERR_ZERO_DIVISION;
    }
    return SB2_OK;
}

int sim_general_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                    int64_t nnz, int min_support, double global_mean, const double* x_biases, const double* y_biases,
                    double shrinkage, int64_t row_begin, int64_t row_end, const int32_t* rows, bool upper,
                    double* sim_out, int64_t out_ld, cudaStream_t st);

__global__ void sim_visits_kernel(int64_t n_y, const int64_t* __restrict__ y_ptr, double* __restrict__ out) {
    const int64_t y = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    double v = 0.0;
    if (y < n_y) {
        const double len = (double)(y_ptr[y + 1] - y_ptr[y]);
        v = len * len;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if ((threadIdx.x & 31) == 0 && v != 0.0) atomicAdd(out, v);
}

// Two implementations of the same four functions:
//   digit   (sim_core above): dense masked contractions on the int8 tensor cores.  Cost ~ accumulators x n_x^2 x n_y,
//           independent of the sparsity; exact for cosine / msd / pearson on grid ratings, 1e-9-class for
//           pearson_baseline; needs non-negative ratings on a 1/d grid and unique (x, y) pairs.
//   general (sim_general.cu): the reference's own loop nest on the CUDA cores, fp64, bit-identical to the reference for
//           ANY input.  Cost ~ sum_y |yr[y]|^2 co-ratings (~2.1e10 / s on a B200 at n_x = 27k).
// rating_denom == 0 (no grid / negative ratings) and duplicated pairs (detected by the pack kernel) always take the
// general path: everything the reference accepts is computed, nothing is rejected.  Otherwise the cheaper one by the
// cost model below runs; pearson_baseline prefers the general path unless the digit path is clearly (1.5x) faster,
// because only the general path reproduces the reference's bits there.  SB2_SIM_PATH=digit|general overrides.
// A row-list build (rows != nullptr, slots [0, row_end)) is costed for its own rows, without symmetry, where both paths
// give the same bits (cosine / msd / pearson on a power-of-two grid: every sum is exact on both).  Elsewhere
// (pearson_baseline, grids like 1/10) it takes the path the full build takes, so that its rows are the full build's
// rows bit for bit.
static int sim_dispatch(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                        int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                        const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end,
                        const int32_t* row_list, double* sim_out, int64_t out_ld, bool upper, cudaStream_t st) {
    if (kind < 0 || kind > 3 || n_x <= 0 || n_y < 0 || row_begin < 0 || (!row_list && row_end > n_x) ||
        (row_list && (row_begin != 0 || upper)) || row_begin >= row_end) {
        set_error("sim_build: invalid argument");
        return SB2_ERR_INVALID;
    }
    if (row_list) {
        DevBuf bad_d;
        SB2_TRY(bad_d.alloc(ST_NWORDS * sizeof(int), st));
        SB2_CUDA(cudaMemsetAsync(bad_d.p, 0, ST_NWORDS * sizeof(int), st));
        sim_check_rows_kernel<<<(unsigned)ceil_div(row_end, 256), 256, 0, st>>>(row_list, row_end, n_x, bad_d.as<int>());
        SB2_LAUNCH_CHECK();
        int bad[ST_NWORDS];
        SB2_CUDA(cudaMemcpyAsync(bad, bad_d.p, sizeof(bad), cudaMemcpyDeviceToHost, st));
        SB2_CUDA(cudaStreamSynchronize(st));
        if (bad[ST_BAD_ROW]) {
            set_error("sim_build_rows: row id out of range for n_x=%lld", (long long)n_x);
            return SB2_ERR_INVALID;
        }
    }
    bool use_digit = rating_denom > 0;
    const char* force = getenv("SB2_SIM_PATH");
    if (force && force[0] == 'g') use_digit = false;
    if (use_digit && !(force && force[0] == 'd') && n_y > 0) {
        DevBuf v_d;
        SB2_TRY(v_d.alloc(sizeof(double), st));
        SB2_CUDA(cudaMemsetAsync(v_d.p, 0, sizeof(double), st));
        sim_visits_kernel<<<(unsigned)ceil_div(n_y, 256), 256, 0, st>>>(n_y, y_ptr, v_d.as<double>());
        SB2_LAUNCH_CHECK();
        double visits = 0.0;
        SB2_CUDA(cudaMemcpyAsync(&visits, v_d.p, sizeof(double), cudaMemcpyDeviceToHost, st));
        SB2_CUDA(cudaStreamSynchronize(st));
        const bool same_bits = kind != SB2_SIM_PEARSON_BASELINE && (rating_denom & (rating_denom - 1)) == 0;
        const bool as_full = row_list && !same_bits;
        const double rows = (double)(as_full ? n_x : row_end - row_begin), frac = rows / (double)n_x;
        // general: co-ratings of the shard's rows + zeroing / reading the 32-byte column records of every row
        const double keep = upper ? 1.0 - ((double)row_begin + 0.5 * rows) / (double)n_x : 1.0;  // columns >= row_begin
        const double t_general = frac * keep * visits / 2.0e10 + rows * (double)n_x * 64.0 / 3.0e12 + 2e-4;
        // digit: accumulators x tiles x k at the measured 3.6 POP/s issued, + packing the dense panels
        const int n_acc = kind == SB2_SIM_PEARSON_BASELINE ? 30 : kind == SB2_SIM_PEARSON ? 6 : 4;
        const double n_pad = (double)round_up(n_x, 256), k_pad = (double)round_up(std::max<int64_t>(n_y, 1), 128);
        const bool tri = as_full || (!row_list && row_begin == 0 && row_end == n_x) || upper;
        const double cols = tri ? (n_pad - (double)row_begin - 0.5 * rows) : n_pad;
        const double t_digit = 2.0 * n_acc * rows * cols * k_pad / 3.6e15 + (n_acc / 2 + 3) * n_pad * k_pad / 4.0e12 + 3e-4;
        const double bias = kind == SB2_SIM_PEARSON_BASELINE ? 1.5 : 1.0;
        use_digit = t_digit * bias < t_general;
    }
    int rc = SB2_ERR_DUPLICATE;
    if (use_digit)
        rc = sim_core(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases, y_biases,
                      shrinkage, row_begin, row_end, row_list, sim_out, out_ld, nullptr, upper, st);
    if (rc != SB2_ERR_DUPLICATE) return rc;
    return sim_general_dev(kind, n_x, n_y, y_ptr, x_idx, r, nnz, min_support, global_mean, x_biases, y_biases, shrinkage,
                           row_begin, row_end, row_list, upper, sim_out, out_ld, st);
}

int sim_build_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                  int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                  const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end, double* sim_out,
                  cudaStream_t st) {
    return sim_dispatch(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases, y_biases,
                        shrinkage, row_begin, row_end, nullptr, sim_out, n_x, false, st);
}

// rows[0 .. n_rows) of the matrix, in the given order (repeats allowed): out[b * ld + j] = sim[rows[b]][j], the bits of
// the same rows of the full build
int sim_build_rows_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                       int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                       const double* y_biases, double shrinkage, const int32_t* rows, int64_t n_rows, double* out,
                       int64_t ld, cudaStream_t st) {
    if (n_rows == 0) return SB2_OK;
    if (!rows || !out || n_rows < 0 || ld < n_x) {
        set_error("sim_build_rows: invalid argument");
        return SB2_ERR_INVALID;
    }
    return sim_dispatch(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases, y_biases,
                        shrinkage, 0, n_rows, rows, out, ld, false, st);
}

// row shard of a symmetric multi-rank build: only sim[i][j] with j >= row_begin is computed (tiles at or above the
// block diagonal, mirrored inside the shard's own diagonal square); the columns before row_begin are the transposes
// of blocks owned by the shards before this one and are left untouched.
int sim_build_upper_dev(int kind, int64_t n_x, int64_t n_y, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                        int64_t nnz, int rating_denom, int min_support, double global_mean, const double* x_biases,
                        const double* y_biases, double shrinkage, int64_t row_begin, int64_t row_end, double* sim_out,
                        cudaStream_t st) {
    return sim_dispatch(kind, n_x, n_y, y_ptr, x_idx, r, nnz, rating_denom, min_support, global_mean, x_biases, y_biases,
                        shrinkage, row_begin, row_end, nullptr, sim_out, n_x, true, st);
}

// SlopeOne.fit (slope_one.pyx:44-80): u_ptr / i_idx / r is the ur CSR (items rated by each user)
int slope_one_fit_dev(int64_t n_items, int64_t n_users, const int64_t* u_ptr, const int32_t* i_idx, const double* r,
                      int64_t nnz, int64_t* freq_out, double* dev_out, cudaStream_t st) {
    if (!freq_out || !dev_out) {
        set_error("slope_one_fit: null output");
        return SB2_ERR_INVALID;
    }
    return sim_core(KIND_SLOPE_ONE, n_items, n_users, u_ptr, i_idx, r, nnz, 1, 0, 0.0, nullptr, nullptr, 0.0, 0, n_items,
                    nullptr, dev_out, n_items, freq_out, false, st);
}

// Smallest supported denominator d such that every rating is an integer multiple of 1/d in [0, 65535/d]
// (1 stars, 2 half-stars, ..., 100 Jester's two decimals); 0 when the ratings are on none of the grids.
// One pass of sim_analyze_kernel per candidate instead of several numpy passes over the ratings on the host.
int rating_denominator_dev(const double* r, int64_t nnz, int* denom_out, cudaStream_t st) {
    static const int cand[] = {1, 2, 4, 5, 10, 20, 100, 1000};
    *denom_out = 1;
    if (nnz <= 0) return SB2_OK;
    DevBuf status_d;
    SB2_TRY(status_d.alloc(ST_NWORDS * sizeof(int), st));
    for (int d : cand) {
        SB2_CUDA(cudaMemsetAsync(status_d.p, 0, ST_NWORDS * sizeof(int), st));
        sim_analyze_kernel<<<(unsigned)ceil_div(nnz, 256), 256, 0, st>>>(r, nnz, (double)d, 0, status_d.as<int>(), nullptr, 0,
                                                                        0.0, nullptr, nullptr);
        SB2_LAUNCH_CHECK();
        int h[ST_NWORDS];
        SB2_CUDA(cudaMemcpyAsync(h, status_d.p, sizeof(h), cudaMemcpyDeviceToHost, st));
        SB2_CUDA(cudaStreamSynchronize(st));
        if (!h[ST_BAD_RATING]) {
            *denom_out = d;
            return SB2_OK;
        }
    }
    *denom_out = 0;
    return SB2_OK;
}

}  // namespace sb2
