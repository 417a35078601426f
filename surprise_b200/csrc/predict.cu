// Batched estimate kernels: factor models (gather + dot) and k-NN (gather + stable top-k select +
// ordered weighted sum).  These replace the per-pair Python estimate() calls that AlgoBase.test makes
// (algo_base.py:191-218 -> matrix_factorization.pyx:269-299 / :506-522 / :737-761, knns.py:99-123 /
// :274-309).
#include "common.cuh"

namespace sb2 {

// ------------------------------------------------------------------------------------------------
// Factor models.  One warp per (u, i) pair; lanes stride the factor dimension, partial dots are
// combined with a shuffle tree (the reference uses np.dot, whose summation order is BLAS-defined, so
// the contract here is fp64 accuracy, not bit equality).
// ------------------------------------------------------------------------------------------------
__global__ void mf_predict_kernel(int64_t n_pairs, const int32_t* __restrict__ u, const int32_t* __restrict__ i, int f,
                                  int biased, double mu, const double* __restrict__ pu, const double* __restrict__ qi,
                                  const double* __restrict__ bu, const double* __restrict__ bi,
                                  const double* __restrict__ yj, const int64_t* __restrict__ u_ptr,
                                  const int32_t* __restrict__ ui_idx, double* __restrict__ est,
                                  uint8_t* __restrict__ impossible) {
    const int lane = threadIdx.x & 31;
    const int64_t k = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (k >= n_pairs) return;
    const int32_t uu = u[k], ii = i[k];
    const bool ku = uu >= 0, ki = ii >= 0;
    double e = 0.0;
    uint8_t imp = 0;
    if (biased) {
        e = mu;
        if (ku) e += bu[uu];
        if (ki) e += bi[ii];
    } else if (!(ku && ki)) {
        imp = 1;  // PredictionImpossible('User and item are unkown.')
    }
    if (ku && ki) {
        const double* p = pu + (size_t)uu * f;
        const double* q = qi + (size_t)ii * f;
        double part = 0.0;
        if (yj) {
            const int64_t b = u_ptr[uu], en = u_ptr[uu + 1];
            const double sq = sqrt((double)(en - b));
            for (int j = lane; j < f; j += 32) {
                double s = 0.0;
                for (int64_t a = b; a < en; ++a) s += yj[(size_t)ui_idx[a] * f + j];
                part += q[j] * (p[j] + s / sq);
            }
        } else {
            for (int j = lane; j < f; j += 32) part += q[j] * p[j];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xFFFFFFFFu, part, o);
        e = biased ? e + part : part;
    }
    if (lane == 0) {
        est[k] = e;
        impossible[k] = imp;
    }
}

int mf_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int f, int biased, double mu, const double* pu,
                   const double* qi, const double* bu, const double* bi, const double* yj, const int64_t* u_ptr,
                   const int32_t* ui_idx, double* est, uint8_t* impossible, cudaStream_t st) {
    if (n_pairs <= 0) return SB2_OK;
    const int threads = 256;
    mf_predict_kernel<<<(unsigned)ceil_div(n_pairs * 32, threads), threads, 0, st>>>(
        n_pairs, u, i, f, biased, mu, pu, qi, bu, bi, yj, u_ptr, ui_idx, est, impossible);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

// ------------------------------------------------------------------------------------------------
// k-NN.  One warp per (x, y) pair.
//   neighbors = [(sim[x, x2], r) for (x2, r) in yr[y]]; heapq.nlargest(k, key=sim)
// heapq.nlargest == sorted(reverse=True)[:k]: descending by sim, ties keep list order, i.e. the total order
// (sim desc, position asc).  Selection:
//   phase A  every lane walks its strided share of the list ONCE (index load + gathered sim) and keeps its own
//            best KNN_L candidates, sorted, in registers -- one pass over the list instead of one per neighbour;
//   phase B  up to k rounds: the best head of the 32 lane buffers is found with three warp reductions
//            (redux.sync on the high / low word of an order-preserving integer image of sim, then on the
//            position), the winning lane advances.  A lane whose buffer runs dry although it had to drop
//            candidates re-walks its share for the next KNN_L after the last one it gave out (exact, rare).
// The weighted sums are accumulated by every lane identically, in selection order, in round-to-nearest fp64
// without contraction -- the same sequence of operations as the reference, hence the same bits.
// ------------------------------------------------------------------------------------------------
constexpr int KNN_WARPS = 8;
constexpr int KNN_L = 8;  // candidates kept per lane

// order-preserving map double -> uint64 (larger = more similar); NaN -> 0 (never selected); -0.0 == +0.0
__device__ __forceinline__ unsigned long long knn_key(double s) {
    if (s != s) return 0ull;
    const unsigned long long b = (unsigned long long)__double_as_longlong(s + 0.0);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double knn_unkey(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    return __longlong_as_double((long long)b);
}

struct KnnBuf {
    unsigned long long key[KNN_L];
    int pos[KNN_L];
    int cnt;       // valid entries
    bool dropped;  // an eligible candidate did not fit: more may follow after the buffer's last entry
};

// lane-local: best KNN_L candidates strictly after (bound_key, bound_pos) in (key desc, pos asc) order
__device__ __forceinline__ void knn_fill(KnnBuf& q, const double* __restrict__ srow, const int32_t* __restrict__ idx,
                                         int64_t len, int lane, bool bounded, unsigned long long bound_key, int bound_pos) {
    q.cnt = 0;
    q.dropped = false;
#pragma unroll
    for (int t = 0; t < KNN_L; ++t) { q.key[t] = 0ull; q.pos[t] = 0x7FFFFFFF; }
    for (int64_t a0 = lane; a0 < len; a0 += 4 * 32) {
        double sv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t a = a0 + 32 * u;
            sv[u] = a < len ? srow[idx[a]] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int64_t a = a0 + 32 * u;
            if (a >= len) break;
            unsigned long long ck = knn_key(sv[u]);
            int cp = (int)a;
            if (ck == 0ull) continue;  // NaN
            if (bounded && !(ck < bound_key || (ck == bound_key && cp > bound_pos))) continue;
            // positions arrive in ascending order, so on equal keys the newcomer is worse: insert below equals
            if (q.cnt == KNN_L && !(ck > q.key[KNN_L - 1])) { q.dropped = true; continue; }
            if (q.cnt == KNN_L) q.dropped = true; else ++q.cnt;
#pragma unroll
            for (int t = 0; t < KNN_L; ++t) {
                const bool better = ck > q.key[t] || (ck == q.key[t] && cp < q.pos[t]);
                if (better) {
                    const unsigned long long tk = q.key[t]; const int tp = q.pos[t];
                    q.key[t] = ck; q.pos[t] = cp;
                    ck = tk; cp = tp;
                }
            }
        }
    }
}

// Short lists (len <= KNN_CAP, k <= KNN_KCAP -- the common case: |yr[y]| is ~10^2): threshold select.
//   1. every lane loads its strided share of the neighbour similarities ONCE into shared memory as order-preserving
//      integer keys (non-positive and NaN similarities can never contribute: key 0);
//   2. the k-th largest key is found by bisection on the key VALUE: count(key >= mid) with one redux.sync.add per
//      step, starting from the [min, max] of the candidates and stopping as soon as a cut with exactly k candidates
//      above it is found -- typically ~10-15 steps, against k rounds of three reductions each;
//   3. the <= k survivors are ranked among themselves in the total order (sim desc, position asc) -- exactly the
//      order heapq.nlargest returns them in -- and the weighted sums are accumulated in that order in round-to-nearest
//      fp64, every lane identically: same operations in the same sequence as the reference, same bits.
constexpr int KNN_CAP = 512;    // candidates per warp held in shared memory
constexpr int KNN_SLOTS = KNN_CAP / 32;
constexpr int KNN_KCAP = 128;   // survivors per warp
constexpr unsigned long long KNN_KEY0 = 0x8000000000000000ull;  // knn_key(0.0)

struct KnnSums {
    double sum_sim, sum_r;
    int ak;
};

// Bisection on 32-bit VALUES held by the lanes (get(slot, v) -> is this slot a member, and its value): finds the largest
// member value `cut` with count(v >= cut) >= kk and that count.  Both ends are snapped to member values after every
// step (lo: the smallest member >= mid, hi: the largest member < mid), so the number of steps is bounded by the number
// of DISTINCT values in the range (msd / pearson on star ratings produce many equal similarities) as well as by the 32
// bits.  Needs lo0 / hi0 = the smallest / largest member value and n0 = the number of members (>= kk).
template <class Get>
__device__ __forceinline__ void knn_bisect32(int n_slots, int kk, unsigned lo, unsigned hi, int n0, Get get, unsigned& cut,
                                             int& n_ge) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    cut = lo;
    n_ge = n0;
    while (lo < hi) {
        const unsigned mid = lo + ((hi - lo) >> 1) + 1;       // lo < mid <= hi
        int c = 0;
        unsigned up = 0xFFFFFFFFu, down = 0u;                 // smallest member >= mid, largest member < mid
        for (int slot = 0; slot < n_slots; ++slot) {
            unsigned v;
            if (get(slot, v)) {
                const bool ge = v >= mid;
                c += ge;
                up = (ge && v < up) ? v : up;
                down = (!ge && v > down) ? v : down;
            }
        }
        c = __reduce_add_sync(FULL, c);
        if (c >= kk) {
            lo = __reduce_min_sync(FULL, up); cut = lo; n_ge = c;   // count(>= lo) is still c
            if (c == kk) break;
        } else {
            hi = __reduce_max_sync(FULL, down);                     // >= lo: count(>= lo) >= kk > c
        }
    }
}

template <class TermFn>
__device__ __forceinline__ KnnSums knn_select_short(const double* __restrict__ srow, const int32_t* __restrict__ idx, int len,
                                                    int k, int lane, unsigned long long* __restrict__ ckey /* [KNN_CAP] */,
                                                    unsigned long long* __restrict__ skey /* [KNN_KCAP] */,
                                                    int* __restrict__ spos /* [2 * KNN_KCAP] */, TermFn term_of) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    const int n_slots = (len + 31) >> 5;   // candidate a = lane + 32 * slot, keys at ckey[slot * 32 + lane]
    // 1. keys of this lane's candidates
    int n_pos = 0;
    unsigned hmax = 0u, hmin = 0xFFFFFFFFu;   // high words of the largest / smallest positive key of this lane
    // eight neighbour indices, then eight gathered similarities, in flight per lane: the gathers are random 8-byte
    // reads of a sim row (one DRAM / L2 sector each) and the kernel waits on them more than on anything else
    constexpr int KNN_MLP = 8;
    for (int slot0 = 0; slot0 < n_slots; slot0 += KNN_MLP) {
        int ia[KNN_MLP];
        double sv[KNN_MLP];
#pragma unroll
        for (int u = 0; u < KNN_MLP; ++u) {
            const int a = lane + 32 * (slot0 + u);
            ia[u] = a < len ? idx[a] : -1;
        }
#pragma unroll
        for (int u = 0; u < KNN_MLP; ++u) sv[u] = ia[u] >= 0 ? srow[ia[u]] : -1.0;
#pragma unroll
        for (int u = 0; u < KNN_MLP; ++u) {
            if (slot0 + u < n_slots) {
                unsigned long long key = knn_key(sv[u]);
                if (key <= KNN_KEY0) key = 0ull;   // sim <= 0 (or NaN): never part of the sums (knns.py:110-113)
                ckey[(slot0 + u) * 32 + lane] = key;
                if (key) {
                    const unsigned h = (unsigned)(key >> 32);
                    ++n_pos; hmax = h > hmax ? h : hmax; hmin = h < hmin ? h : hmin;
                }
            }
        }
    }
    n_pos = __reduce_add_sync(FULL, n_pos);
    KnnSums out{0.0, 0.0, 0};
    if (n_pos == 0) return out;
    const int kk = n_pos < k ? n_pos : k;
    // 2. cut: the largest candidate key T with count(key >= T) >= kk.  The keys are 64 bits wide but almost always
    //    differ in their HIGH words (sign, exponent, 20 mantissa bits), or not at all (equal similarities): the
    //    bisection runs on the high words (32-bit compares and single warp reductions); only when several DIFFERENT keys
    //    share the high word of the k-th one does a second bisection on the low words of that group follow.
    unsigned long long cut = 1ull;   // n_pos <= k: every positive candidate survives
    int n_ge = n_pos;
    int n_eq_keep = 0x7FFFFFFF;      // candidates equal to `cut` that survive (in position order)
    if (n_pos > kk) {
        __syncwarp(FULL);            // the keys of all lanes are in shared memory
        const unsigned* chi = reinterpret_cast<const unsigned*>(ckey) + 1;   // high word of ckey[j]: chi[2 j]
        const unsigned lo_h0 = __reduce_min_sync(FULL, hmin), hi_h0 = __reduce_max_sync(FULL, hmax);
        unsigned cut_h;
        int n_ge_h;
        // non-positive candidates have key 0: never >= mid (> lo_h0 > 0), never the largest value below mid
        knn_bisect32(n_slots, kk, lo_h0, hi_h0, n_pos,
                     [&](int slot, unsigned& v) { v = chi[2 * (slot * 32 + lane)]; return true; }, cut_h, n_ge_h);
        if (n_ge_h == kk) {
            // exactly kk candidates have a high word >= cut_h: they are the survivors, whatever their low words
            cut = ((unsigned long long)cut_h << 32) - 1ull;
            n_ge = kk;
            n_eq_keep = 0;           // (a stray key equal to cut itself has the high word cut_h - 1: not a survivor)
        } else {
            // the group with high word cut_h holds the k-th key: how many lie above it, and the range of its low words
            int c_gt = 0, c_eq = 0;
            unsigned lmin = 0xFFFFFFFFu, lmax = 0u;
            for (int slot = 0; slot < n_slots; ++slot) {
                const unsigned long long key = ckey[slot * 32 + lane];
                const unsigned h = (unsigned)(key >> 32), l = (unsigned)key;
                c_gt += h > cut_h;
                if (h == cut_h) { ++c_eq; lmin = l < lmin ? l : lmin; lmax = l > lmax ? l : lmax; }
            }
            c_gt = __reduce_add_sync(FULL, c_gt);
            c_eq = __reduce_add_sync(FULL, c_eq);
            lmin = __reduce_min_sync(FULL, lmin);
            lmax = __reduce_max_sync(FULL, lmax);
            unsigned cut_l = lmin;
            int n_ge_l = c_eq;
            if (lmin != lmax)   // different keys in the group: the (kk - c_gt)-th largest low word
                knn_bisect32(n_slots, kk - c_gt, lmin, lmax, c_eq,
                             [&](int slot, unsigned& v) {
                                 const unsigned long long key = ckey[slot * 32 + lane];
                                 v = (unsigned)key;
                                 return (unsigned)(key >> 32) == cut_h;
                             }, cut_l, n_ge_l);
            cut = ((unsigned long long)cut_h << 32) | cut_l;
            n_ge = c_gt + n_ge_l;
        }
    }
    // 3. survivors: key > cut all; key == cut in position order until kk are there (heapq.nlargest keeps list order
    //    among equal keys), i.e. the n_ge - kk LAST candidates equal to `cut` are left out
    if (n_ge > kk) {
        int c_gt = 0;
        for (int slot = 0; slot < n_slots; ++slot) c_gt += ckey[slot * 32 + lane] > cut;
        n_eq_keep = kk - __reduce_add_sync(FULL, c_gt);
    }
    // compaction in position order (slot-major, lane-minor = ascending position)
    int base = 0, eq_seen = 0;
    for (int slot = 0; slot < n_slots; ++slot) {
        const unsigned long long key = ckey[slot * 32 + lane];
        const bool eq = key == cut, gt = key > cut;
        const unsigned below = (1u << lane) - 1u;
        const unsigned m_eq = __ballot_sync(FULL, eq);
        const bool take = gt || (eq && eq_seen + __popc(m_eq & below) < n_eq_keep);
        const unsigned m = __ballot_sync(FULL, take);
        if (take) {
            const int o = base + __popc(m & below);
            skey[o] = key & 0x7FFFFFFFFFFFFFFFull;   // survivors are positive: the similarity's own bits
            spos[o] = lane + 32 * slot;
        }
        base += __popc(m);
        eq_seen += __popc(m_eq);
    }
    __syncwarp(FULL);
    // Rank of every survivor in (sim desc, pos asc) -- survivors are in ascending position, so among equal similarities
    // the earlier index wins; the ranks are a permutation of 0 .. kk-1.  The lane that ranks a survivor also computes
    // its term of the weighted sum and drops (sim, term) at its rank into bt[] (the candidate keys are dead by now).
    // Survivors are positive, so their similarities compare as doubles (one DSETP instead of a two-word integer compare).
    double2* bt = reinterpret_cast<double2*>(ckey);
    const double* ssim = reinterpret_cast<const double*>(skey);
    auto place = [&](int j, int rank, double sj) { bt[rank] = make_double2(sj, term_of(sj, spos[j])); };
    if (kk <= 48) {
        // lane -> survivor `lane` against all kk; survivors 32 .. kk-1 (k = 40, the reference's default: eight of them)
        // are ranked by `parts` lanes each, every one counting a slice of the survivors
        const int ja = lane;
        const double sa = ja < kk ? ssim[ja] : 0.0;
        int ra = 0;
        for (int t = 0; t < kk; ++t) {
            const double st = ssim[t];
            ra += (st > sa) || (st == sa && t < ja);
        }
        if (ja < kk) place(ja, ra, sa);
        if (kk > 32) {
            const int per = kk <= 40 ? 8 : 16, parts = 32 / per;
            const int jb = 32 + (lane % per), q = lane / per;
            const double sb = jb < kk ? ssim[jb] : 0.0;
            const int chunk = (kk + parts - 1) / parts, t0 = q * chunk;
            int rb = 0;
            for (int i = 0; i < chunk; ++i) {
                const int t = t0 + i;
                if (t < kk) {
                    const double st = ssim[t];
                    rb += (st > sb) || (st == sb && t < jb);
                }
            }
            for (int o = per; o < 32; o <<= 1) rb += __shfl_xor_sync(FULL, rb, o);
            if (q == 0 && jb < kk) place(jb, rb, sb);
        }
    } else {
        for (int j0 = 0; j0 < kk; j0 += 64) {   // lane handles survivors j0 + lane and j0 + 32 + lane in one sweep
            const int ja = j0 + lane, jb = j0 + 32 + lane;
            const double sa = ja < kk ? ssim[ja] : 0.0, sb = jb < kk ? ssim[jb] : 0.0;
            int ra = 0, rb = 0;
            for (int t = 0; t < kk; ++t) {
                const double st = ssim[t];
                ra += (st > sa) || (st == sa && t < ja);
                rb += (st > sb) || (st == sb && t < jb);
            }
            if (ja < kk) place(ja, ra, sa);
            if (jb < kk) place(jb, rb, sb);
        }
    }
    __syncwarp(FULL);
    // ordered sums: every lane folds the kk (sim, term) pairs in selection order (one 16-byte broadcast read each)
#pragma unroll 4
    for (int t = 0; t < kk; ++t) {
        const double2 v = bt[t];
        out.sum_sim = __dadd_rn(out.sum_sim, v.x);
        out.sum_r = __dadd_rn(out.sum_r, v.y);
    }
    out.ak = kk;
    __syncwarp(FULL);   // the buffers are reused by this warp's next pair
    return out;
}

// Long lists (len > KNN_CAP) or very large k: lane-local sorted buffers + one selection round per neighbour (see the
// header comment of this section).  Kept out of line: its register needs must not cap the short path's occupancy.
template <class TermFn>
__device__ __noinline__ KnnSums knn_select_long(const double* __restrict__ srow, const int32_t* __restrict__ idx, int64_t len,
                                    int k, int lane, unsigned long long* __restrict__ bkey /* [KNN_L][32] */,
                                    int* __restrict__ bpos /* [KNN_L][32] */, TermFn term_of) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    double sum_sim = 0.0, sum_r = 0.0;
    int ak = 0;
    KnnBuf q;
    knn_fill(q, srow, idx, len, lane, false, 0ull, 0);
    // the sorted lane buffers live in shared memory ([slot][lane]: conflict-free) so that the head is one
    // indexed read per round instead of a select chain over registers (the kernel is issue-bound)
#pragma unroll
    for (int u = 0; u < KNN_L; ++u) { bkey[u * 32 + lane] = q.key[u]; bpos[u * 32 + lane] = q.pos[u]; }
    int head = 0;
    const int64_t rounds = len < (int64_t)k ? len : (int64_t)k;
    // Selection runs in batches of 32 rounds that touch only registers; lane j keeps the j-th winner of the
    // batch.  The ratings (and neighbour baselines) of a batch are then gathered by all lanes at once and the
    // two sums advance in selection order from lane 0 upwards -- one memory round trip per batch instead
    // of one per neighbour in the dependent chain.
    bool done = false;
    for (int64_t t0 = 0; t0 < rounds && !done; t0 += 32) {
        const int batch = (int)((rounds - t0) < 32 ? (rounds - t0) : 32);
        int nb = 0;
        double my_bs = 0.0;
        int my_bp = 0;
        for (int t = 0; t < batch; ++t) {
            // refill lanes that ran dry but had dropped candidates (the bound is the last entry they gave out)
            const bool dry = head == q.cnt && q.dropped;
            if (__any_sync(FULL, dry)) {
                if (dry) {
                    const unsigned long long bk = bkey[(KNN_L - 1) * 32 + lane];
                    const int bp = bpos[(KNN_L - 1) * 32 + lane];
                    knn_fill(q, srow, idx, len, lane, true, bk, bp);
#pragma unroll
                    for (int u = 0; u < KNN_L; ++u) { bkey[u * 32 + lane] = q.key[u]; bpos[u * 32 + lane] = q.pos[u]; }
                    head = 0;
                }
                __syncwarp(FULL);
            }
            // head of this lane's buffer (entries are kept best-first)
            unsigned long long hk = 0ull;
            int hp = 0x7FFFFFFF;
            if (head < q.cnt) { hk = bkey[head * 32 + lane]; hp = bpos[head * 32 + lane]; }
            const unsigned hi = (unsigned)(hk >> 32);
            const unsigned m_hi = __reduce_max_sync(FULL, hi);
            bool alive = hi == m_hi && hk != 0ull;
            const unsigned lo = alive ? (unsigned)hk : 0u;
            const unsigned m_lo = __reduce_max_sync(FULL, lo);
            alive = alive && lo == m_lo;
            const unsigned long long bk = ((unsigned long long)m_hi << 32) | m_lo;
            if (bk == 0ull) { done = true; break; }  // nothing (or only NaNs) left
            const int bp = __reduce_min_sync(FULL, alive ? hp : 0x7FFFFFFF);
            const double bs = knn_unkey(bk);
            if (!(bs > 0.0)) { done = true; break; }  // everything that follows is <= 0 and contributes nothing
            if (alive && hp == bp) ++head;
            if (lane == nb) { my_bs = bs; my_bp = bp; }
            ++nb;
        }
        const double term = lane < nb ? term_of(my_bs, my_bp) : 0.0;
        for (int j = 0; j < nb; ++j) {
            sum_sim = __dadd_rn(sum_sim, __shfl_sync(FULL, my_bs, j));
            sum_r = __dadd_rn(sum_r, __shfl_sync(FULL, term, j));
        }
        ak += nb;
    }
    __syncwarp(FULL);
    return KnnSums{sum_sim, sum_r, ak};
}

#ifndef SB2_KNN_MIN_BLOCKS
#define SB2_KNN_MIN_BLOCKS 4
#endif
__global__ void __launch_bounds__(KNN_WARPS * 32, SB2_KNN_MIN_BLOCKS)
knn_predict_kernel(int64_t n_pairs, const int32_t* __restrict__ x, const int32_t* __restrict__ y, int64_t n_x,
                   const double* __restrict__ sim, int64_t sim_ld, const int32_t* __restrict__ sim_row,
                   const int64_t* __restrict__ y_ptr,
                   const int32_t* __restrict__ x_idx, const double* __restrict__ r, int k, int min_k, int mode,
                   double mu, const double* __restrict__ bx, const double* __restrict__ by, double* __restrict__ est,
                   int32_t* __restrict__ actual_k, uint8_t* __restrict__ impossible) {
    constexpr unsigned FULL = 0xFFFFFFFFu;
    // long-list path: sorted lane buffers [KNN_L][32] of keys / positions.  Short-list path: candidate keys
    // [KNN_SLOTS][32] (their head is reused for the sorted survivor keys), survivor keys, survivor positions
    // (first half: in position order, second half: sorted)
    __shared__ __align__(16) unsigned long long bkey_s[KNN_WARPS][KNN_CAP];
    __shared__ int bpos_s[KNN_WARPS][KNN_L * 32 > 2 * KNN_KCAP ? KNN_L * 32 : 2 * KNN_KCAP];
    __shared__ unsigned long long skey_s[KNN_WARPS][KNN_KCAP];
    static_assert(KNN_KCAP <= KNN_CAP && KNN_L * 32 <= KNN_CAP, "buffer reuse");
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int64_t p = blockIdx.x * (int64_t)KNN_WARPS + w; p < n_pairs; p += (int64_t)gridDim.x * KNN_WARPS) {
        const int32_t xx = x[p], yy = y[p];
        const bool kx = xx >= 0, ky = yy >= 0;
        double e = 0.0;
        int ak = -1;
        uint8_t imp = 0;
        if (mode == 1 || mode == 2) {
            e = mu;
            // est += bu[u] first, then bi[i] (knns.py:276-280); mode 1: x is the user, mode 2: y is
            if (mode == 1) { if (kx) e = __dadd_rn(e, bx[xx]); if (ky) e = __dadd_rn(e, by[yy]); }
            else { if (ky) e = __dadd_rn(e, by[yy]); if (kx) e = __dadd_rn(e, bx[xx]); }
        }
        if (!(kx && ky)) {
            if (mode == 0 || mode >= 3) imp = 1;  // KNNBasic / WithMeans / WithZScore raise PredictionImpossible
        } else {
            if (mode >= 3) e = bx[xx];  // means[x] (knns.py:187, :382)
            const int64_t b = y_ptr[yy], len = y_ptr[yy + 1] - b;
            const double* srow = sim + (size_t)sim_row[p] * (size_t)sim_ld;  // row x of the matrix
            const int32_t* idx = x_idx + b;
            // per-neighbour term of the weighted sum (knns.py:113 / :195 / :296-297 / :389)
            auto term_of = [&](double bs, int pos) -> double {
                const double rr = r[b + pos];
                if (mode == 0) return __dmul_rn(bs, rr);
                const int32_t nbr = idx[pos];
                if (mode == 3) return __dmul_rn(bs, __dsub_rn(rr, bx[nbr]));
                if (mode == 4) return __ddiv_rn(__dmul_rn(bs, __dsub_rn(rr, bx[nbr])), by[nbr]);
                const double nb_bsl = __dadd_rn(__dadd_rn(mu, bx[nbr]), by[yy]);
                return __dmul_rn(bs, __dsub_rn(rr, nb_bsl));
            };
            double sum_sim = 0.0, sum_r = 0.0;
            ak = 0;
            if (len <= KNN_CAP && k <= KNN_KCAP) {
                const KnnSums o = knn_select_short(srow, idx, (int)len, k, lane, bkey_s[w], skey_s[w], bpos_s[w], term_of);
                sum_sim = o.sum_sim; sum_r = o.sum_r; ak = o.ak;
            } else {
                const KnnSums o = knn_select_long(srow, idx, len, k, lane, bkey_s[w], bpos_s[w], term_of);
                sum_sim = o.sum_sim; sum_r = o.sum_r; ak = o.ak;
            }
            if (mode != 0) {
                if (ak < min_k) sum_r = 0.0;
                if (ak > 0) {  // ZeroDivisionError swallowed otherwise
                    if (mode == 4) e = __dadd_rn(e, __dmul_rn(__ddiv_rn(sum_r, sum_sim), by[xx]));
                    else e = __dadd_rn(e, __ddiv_rn(sum_r, sum_sim));
                }
            } else {
                if (ak < min_k) imp = 1;       // PredictionImpossible('Not enough neighbors.')
                else if (ak == 0) imp = 2;     // min_k <= 0: the reference divides 0 / 0
                else e = __ddiv_rn(sum_r, sum_sim);
            }
        }
        if (lane == 0) {
            est[p] = e;
            actual_k[p] = ak;
            impossible[p] = imp;
        }
    }
}

// pair p reads its similarities from sim + sim_row[p] * sim_ld (sim_row = x for the whole matrix)
int knn_predict_dev(int64_t n_pairs, const int32_t* x, const int32_t* y, int64_t n_x, const double* sim,
                    int64_t sim_ld, const int32_t* sim_row, const int64_t* y_ptr, const int32_t* x_idx, const double* r,
                    int k, int min_k, int mode, double mu, const double* bx, const double* by, double* est,
                    int32_t* actual_k, uint8_t* impossible, cudaStream_t st) {
    if (n_pairs <= 0) return SB2_OK;
    if (mode < 0 || mode > 4 || (mode != 0 && !bx) || ((mode == 1 || mode == 2 || mode == 4) && !by)) {
        set_error("knn_predict: invalid mode / missing baselines");
        return SB2_ERR_INVALID;
    }
    int64_t blocks = ceil_div(n_pairs, KNN_WARPS);
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    knn_predict_kernel<<<(unsigned)blocks, KNN_WARPS * 32, 0, st>>>(n_pairs, x, y, n_x, sim, sim_ld, sim_row, y_ptr, x_idx,
                                                                    r, k, min_k, mode, mu, bx, by, est, actual_k,
                                                                    impossible);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

// ------------------------------------------------------------------------------------------------
// SlopeOne.estimate (slope_one.pyx:82-97).  One warp per (u, i):
//   Ri = [j for (j, _) in ur[u] if freq[i, j] > 0];  est = user_mean[u] + sum(dev[i, j] for j in Ri) / len(Ri)
// Python's sum() adds left to right in ur[u] order; lanes gather 32 entries of row i at a time and the
// warp folds them in lane order (every lane performs the same additions), so the bits match.
// ------------------------------------------------------------------------------------------------
__global__ void slope_one_predict_kernel(int64_t n_pairs, const int32_t* __restrict__ u, const int32_t* __restrict__ i,
                                         int64_t n_items, const int64_t* __restrict__ freq,
                                         const double* __restrict__ dev, const int64_t* __restrict__ u_ptr,
                                         const int32_t* __restrict__ i_idx, const double* __restrict__ user_mean,
                                         double* __restrict__ est, uint8_t* __restrict__ impossible) {
    const int lane = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t p = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5; p < n_pairs; p += nwarps) {
        const int32_t uu = u[p], ii = i[p];
        double e = 0.0;
        uint8_t imp = 0;
        if (uu < 0 || ii < 0) {
            imp = 1;  // PredictionImpossible('User and/or item is unkown.')
        } else {
            const int64_t b = u_ptr[uu], len = u_ptr[uu + 1] - b;
            const int64_t* frow = freq + (size_t)ii * (size_t)n_items;
            const double* drow = dev + (size_t)ii * (size_t)n_items;
            double sum = 0.0;
            int64_t cnt = 0;
            for (int64_t a0 = 0; a0 < len; a0 += 32) {
                const int64_t a = a0 + lane;
                bool rel = false;
                double d = 0.0;
                if (a < len) {
                    const int32_t j = i_idx[b + a];
                    rel = frow[j] > 0;
                    if (rel) d = drow[j];
                }
                const unsigned m = __ballot_sync(0xFFFFFFFFu, rel);
                cnt += __popc(m);
                for (unsigned rest = m; rest; rest &= rest - 1) {
                    const int src = __ffs(rest) - 1;
                    sum = __dadd_rn(sum, __shfl_sync(0xFFFFFFFFu, d, src));
                }
            }
            e = user_mean[uu];
            if (cnt > 0) e = __dadd_rn(e, __ddiv_rn(sum, (double)cnt));
        }
        if (lane == 0) {
            est[p] = e;
            impossible[p] = imp;
        }
    }
}

int slope_one_predict_dev(int64_t n_pairs, const int32_t* u, const int32_t* i, int64_t n_items, const int64_t* freq,
                          const double* dev, const int64_t* u_ptr, const int32_t* i_idx, const double* user_mean,
                          double* est, uint8_t* impossible, cudaStream_t st) {
    if (n_pairs <= 0) return SB2_OK;
    int64_t blocks = ceil_div(n_pairs * 32, 256);
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    slope_one_predict_kernel<<<(unsigned)blocks, 256, 0, st>>>(n_pairs, u, i, n_items, freq, dev, u_ptr, i_idx, user_mean,
                                                              est, impossible);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

// ------------------------------------------------------------------------------------------------
// AlgoBase.get_neighbors (algo_base.py:303-334): others = [(x, sim[iid, x]) for x != iid];
// others.sort(key = sim, reverse = True)  -- stable, so ties keep ascending x -- and the first k ids.
// One block per requested row; k rounds of "best element strictly after the previous pick in
// (sim desc, x asc) order", block-wide arg-max through warp shuffles + one shared-memory stage.
// ------------------------------------------------------------------------------------------------
constexpr int TOPK_THREADS = 1024;

__global__ void __launch_bounds__(TOPK_THREADS)
row_topk_kernel(const double* __restrict__ sim, int64_t sim_ld, int64_t n_x, const int32_t* __restrict__ rows, int k,
                int32_t* __restrict__ out) {
    __shared__ double ws[32];
    __shared__ int wi[32];
    __shared__ double pick_s;
    __shared__ int pick_i;
    const int32_t row = rows[blockIdx.x];
    int32_t* o = out + (size_t)blockIdx.x * k;
    if (row < 0 || row >= n_x) {
        for (int t = threadIdx.x; t < k; t += blockDim.x) o[t] = -1;
        return;
    }
    const double* srow = sim + (size_t)row * (size_t)sim_ld;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    double last_s = 0.0;
    int last_i = -1;
    for (int t = 0; t < k; ++t) {
        double bs = 0.0;
        int bi = -1;
        for (int64_t x = threadIdx.x; x < n_x; x += blockDim.x) {
            if (x == row) continue;
            const double s = srow[x];
            const bool after = last_i < 0 || s < last_s || (s == last_s && x > last_i);
            if (after && (bi < 0 || s > bs)) { bs = s; bi = (int)x; }  // ascending x: first max wins
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double os = __shfl_xor_sync(0xFFFFFFFFu, bs, off);
            const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, off);
            if (oi >= 0 && (bi < 0 || os > bs || (os == bs && oi < bi))) { bs = os; bi = oi; }
        }
        if (lane == 0) { ws[w] = bs; wi[w] = bi; }
        __syncthreads();
        if (w == 0) {
            bs = lane < (blockDim.x >> 5) ? ws[lane] : 0.0;
            bi = lane < (blockDim.x >> 5) ? wi[lane] : -1;
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const double os = __shfl_xor_sync(0xFFFFFFFFu, bs, off);
                const int oi = __shfl_xor_sync(0xFFFFFFFFu, bi, off);
                if (oi >= 0 && (bi < 0 || os > bs || (os == bs && oi < bi))) { bs = os; bi = oi; }
            }
            if (lane == 0) { pick_s = bs; pick_i = bi; o[t] = bi; }
        }
        __syncthreads();
        last_s = pick_s;
        last_i = pick_i;
        if (last_i < 0) {  // fewer than k other entries (or only NaNs left): pad with -1
            for (int r = t + 1 + threadIdx.x; r < k; r += blockDim.x) o[r] = -1;
            return;
        }
    }
}

int get_neighbors_dev(int64_t n_x, const double* sim, int64_t sim_ld, int64_t n_rows, const int32_t* rows, int k,
                      int32_t* out, cudaStream_t st) {
    if (n_rows <= 0 || k <= 0) return SB2_OK;
    if (!sim || !rows || !out || sim_ld < n_x) {
        set_error("get_neighbors: invalid argument");
        return SB2_ERR_INVALID;
    }
    row_topk_kernel<<<(unsigned)n_rows, TOPK_THREADS, 0, st>>>(sim, sim_ld, n_x, rows, k, out);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

}  // namespace sb2
