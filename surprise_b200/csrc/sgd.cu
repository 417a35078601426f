// Stratified (DSGD) SGD for SVD -- replaces SVD.sgd (matrix_factorization.pyx:241-262).
//
// The reference walks all_ratings() sequentially; every update reads the latest pu[u], qi[i], so two
// ratings can run concurrently only if they share neither user nor item.  We therefore block the
// rating matrix B x B (B = one persistent CTA per SM): user u lives in user block u % B, item i in
// item block i % B.  An epoch is B strata; in stratum s CTA `ub` owns user block ub (its pu/bu rows
// stay in shared memory for the whole fit) and item block (ub + s) % B, whose qi/bi rows it pulls
// into shared memory, updates, and writes back.  Item blocks move CTA -> CTA along a ring, so instead
// of a grid-wide barrier per stratum each CTA waits on a per-item-block step counter that its ring
// neighbour publishes (st.release / ld.acquire) -- every block is touched by exactly one CTA at a time.
//
// Inside a (user block, item block) cell the ratings form a bipartite multigraph; a greedy edge
// colouring (done once, on the device, at plan creation) splits them into "waves": no two ratings of a
// wave share a user or an item, so the W lane-groups of the CTA process a wave concurrently and
// waves are separated by __syncthreads().  The number of waves is the cell's maximum degree (up to a
// factor < 2), i.e. the inherent sequential depth of the cell.  Colours >= 63 (very popular items)
// fall into a tail that one lane-group replays sequentially.  The schedule is conflict-free by
// construction: no atomics on factors, and the result is deterministic.
//
// One lane-group (G = 4..32 lanes, chosen from n_factors) performs one rating update: 128-bit loads
// of the pu / qi rows, shuffle-tree dot product, bias update by the group leader, factor update and
// 128-bit stores.  Arithmetic is fp32 (the contract is held-out RMSE within 0.005 of the reference).
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <stdlib.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace sb2 {

constexpr int NW = 64;  // waves per cell: 63 colours + 1 sequential tail

struct DsgdArgs {
    int n_users, n_items, B, W, f, FP;  // FP = n_factors rounded up to 4
    int max_ul, max_il;                 // rows per user / item block (ceil)
    int US;                             // user row stride: FP (SVD) or 3*FP (SVD++: [p | z | g], see below)
    int C;                              // CTAs per thread-block cluster (1 = no clusters); B = K * C
    int ibuf;                           // floats per item-block buffer in shared memory
    int s_begin, s_end;                 // strata of this launch, s = T * C + t (SVD: all B; SVD++: one chunk of them)
    int rec_cap;                        // records of a cell staged in shared memory
    const int* ul;                      // records grouped by cell (stratum-major), colour-sorted inside a cell
    const int* il;
    const float* r;
    const int* cell_off;                // B*B + 1 offsets into the records, cell = s * B + user_block
    const int* wave_off;                // [B*B][NW + 1] wave boundaries relative to the cell start
    const int* dep;                     // dependency-driven cells (DEP kernels): per record, the number of earlier
                                        // records of the cell on the same user row | (same item row) << 16
    int dep_sync;                       // experiment: how a DEP warp publishes its row versions (see the kernel)
    float* pu;                          // n_users x FP
    float* qi;                          // n_items x FP
    float* bu;
    float* bi;
    const float* isq;                   // SVD++: 1/sqrt(|I_u|) per user
    float* cnt;                         // SVD++: ratings of u processed since the last y_j application
    int* flags;                         // B step counters (ring hand-off of item blocks)
    float mu, lr_bu, lr_bi, lr_pu, lr_qi, reg_bu, reg_bi, reg_pu, reg_qi, lr_yj, reg_yj;
    int n_epochs;
    long long* prof;                    // optional: [CTA][8]: cycles in {ring wait, block load, updates, write-back, group-0 updates}, #group-0 updates, #waves, 0
    int* status;                        // != 0: a wait ran into its deadline (a CTA / a peer rank was never scheduled)
    int bulk_hop;                       // DSMEM hop as one cp.async.bulk (1) or as per-lane st.shared::cluster (0)
    // ---- ring over P ranks (one process per GPU; P == 1: everything below is unused) --------------------------
    // Rank g owns the users u % P == g for the whole fit and, during sub-epoch E (counted from the start of the
    // fit), the item super-block (g + E) % P, whose (qi, bi) rows live in ring_qi / ring_bi[E & 1].  The CTA that
    // finishes an item block in the last stratum of a sub-epoch stores it straight into the LEFT neighbour's
    // buffer (E + 1) & 1 over NVLink (peer-mapped pointers) and publishes it with a system-scope release on the
    // neighbour's rflags; the neighbour returns a credit once it has consumed the slot it is about to lose.
    int P, rank, E_base;                // E_base: sub-epochs done by earlier launches (SVD++ launches once per epoch)
    int n_items_glob;                   // items of super-block sb: (n_items_glob - sb + P - 1) / P
    float* ring_qi[2];
    float* ring_bi[2];
    float* left_qi[2];                  // the left neighbour's ring buffers (rank - 1)
    float* left_bi[2];
    int* rflags;                        // [B] written by the RIGHT neighbour: sub-epochs whose block it has delivered
    int* left_rflags;
    int* credit;                        // [B] written by the LEFT neighbour: sub-epochs of that block it has consumed
    int* right_credit;
};

__device__ __forceinline__ int ld_relaxed(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_acquire() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ int ld_relaxed_sys(const int* p) {
    int v;
    asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_acquire_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }
__device__ __forceinline__ void st_release_sys(int* p, int v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Every wait of the persistent kernel is bounded: if a partner CTA (or a peer rank) is never scheduled -- SMs held
// by another persistent kernel, an MPS peer, a rank that died -- the waiter gives up after SPIN_LIMIT cycles, raises
// *status and stops waiting for anything else, so the launch drains and the host reports SB2_ERR_CUDA instead of a
// hung GPU.  The clock and *status are looked at once every 256 polls only.
constexpr long long SPIN_LIMIT = 12ll << 30;  // ~6.5 s at 1.97 GHz
struct SpinGuard {
    int* status;
    bool dead;
    __device__ __forceinline__ bool expired(unsigned& polls, long long& t0) {
        if ((++polls & 255u) != 0) return false;
        if (t0 == 0) { t0 = clock64(); return false; }
        if (*reinterpret_cast<volatile int*>(status) != 0 || clock64() - t0 > SPIN_LIMIT) {
            atomicExch(status, 1);
            dead = true;
            return true;
        }
        return false;
    }
};
enum { WAIT_EQ_GPU = 0, WAIT_GE_SYS = 1 };
template <int MODE>
__device__ __forceinline__ void wait_counter(SpinGuard& g, const int* p, int want) {
    if (g.dead) return;
    unsigned polls = 0;
    long long t0 = 0;
    if (MODE == WAIT_EQ_GPU) {
        while (ld_relaxed(p) != want)
            if (g.expired(polls, t0)) return;
        fence_acquire();  // relaxed polls + one acquire fence: no L1 invalidation per poll
    } else {
        while (ld_relaxed_sys(p) < want)
            if (g.expired(polls, t0)) return;
        fence_acquire_sys();
    }
}

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t dsmem_addr(const void* local_smem, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;"
                 : "=r"(r)
                 : "r"((uint32_t)__cvta_generic_to_shared(local_smem)), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ void mbar_init_cta(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count));
}
// arrive on an mbarrier that lives in ANOTHER CTA of the cluster (address from mapa), release at cluster scope
__device__ __forceinline__ void mbar_arrive_remote(uint32_t remote_bar) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
// relaxed arrival on a remote mailbox: the caller has already issued ONE fence.acq_rel.cluster that covers both of
// the hop's arrivals (two release arrivals cost two MEMBARs back to back)
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t remote_bar) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t"
        "}"
        : "=r"(ok)
        : "r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// CTA-scope wait (the default semantics): all that TMA-style consumers need -- the bytes a bulk copy completes on the
// mailbox are visible to the waiting CTA once the phase completes.  No L1 invalidation (CCTL.IVALL) as after a
// cluster-scope acquire.
__device__ __forceinline__ bool mbar_try_wait_cta(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, P1;\n\t"
        "}"
        : "=r"(ok)
        : "r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait_cta(SpinGuard& g, uint64_t* bar, uint32_t parity) {
    if (g.dead) return;
    unsigned polls = 0;
    long long t0 = 0;
    while (!mbar_try_wait_cta(bar, parity))
        if (g.expired(polls, t0)) return;
}
__device__ __forceinline__ void mbar_wait_cluster(SpinGuard& g, uint64_t* bar, uint32_t parity) {
    if (g.dead) return;
    unsigned polls = 0;
    long long t0 = 0;
    while (!mbar_try_wait_cluster(bar, parity))
        if (g.expired(polls, t0)) return;
}
// this CTA's own arrival on one of its mailboxes + the bytes an incoming bulk copy will complete on it
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)),
                 "r"(bytes)
                 : "memory");
}
// generic-proxy writes to shared memory (the updates of this stratum) become visible to the async proxy (bulk copy)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one asynchronous copy of `bytes` (multiple of 16) from this CTA's shared memory into a neighbour's, completing
// on the NEIGHBOUR's mailbox (complete_tx): the copy engine moves the block, no thread of this CTA touches it
__device__ __forceinline__ void dsmem_bulk_push(uint32_t remote_dst, const void* local_src, uint32_t bytes,
                                                uint32_t remote_bar) {
    asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     remote_dst),
                 "r"((uint32_t)__cvta_generic_to_shared(local_src)), "r"(bytes), "r"(remote_bar)
                 : "memory");
}
__device__ __forceinline__ void dsmem_st4(uint32_t addr, float4 v) {
    asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

__device__ __forceinline__ int ld_acquire_cta_shared(const int* p) {
    int v;
    asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_cta_shared(int* p, int v) {
    asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src)
                 : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <bool SMEM>
__device__ __forceinline__ float4 row_ld4(const float* p) {
    if (SMEM) return *reinterpret_cast<const float4*>(p);
    return __ldcg(reinterpret_cast<const float4*>(p));
}
template <bool SMEM>
__device__ __forceinline__ void row_st4(float* p, float4 v) {
    if (SMEM) *reinterpret_cast<float4*>(p) = v;
    else __stcg(reinterpret_cast<float4*>(p), v);
}
template <bool SMEM>
__device__ __forceinline__ float sc_ld(const float* p) {
    if (SMEM) return *p;
    return __ldcg(p);
}
template <bool SMEM>
__device__ __forceinline__ void sc_st(float* p, float v) {
    if (SMEM) *p = v;
    else __stcg(p, v);
}

// one rating update by a group of G lanes (all lanes hold the same ul / il / r).
// CH > 0 (fast path): lane gl owns the 128-bit chunks gl, gl + G, .., gl + (CH - 1) G of the rows and keeps them in
// registers between the dot product and the update.  (G, CH) are chosen so that (CH - 1) G < F4 <= CH G: only the
// last chunk can be ragged, every other load / store is unconditional.  Lanes carrying a dummy rating
// (valid == false, row 0) run the same instruction stream with their stores predicated off, so warps stay
// converged and the shuffles use the full mask.
// CH == 0: 32 lanes stride over the chunks and re-read the rows (rows longer than 256 floats).
// PP (SVD++): the user row is [p | z | g]: z = sum_{j in I_u} y_j / sqrt|I_u| as of the last y_j application,
// advanced by the user's own updates (z += lr_yj (err q - reg_yj z), which is exactly what the reference's
// per-rating y_j updates do to that sum); g accumulates err * q / sqrt|I_u| for the next y_j application.
template <int G, int CH, bool SU, bool SI, bool BIASED, bool PP>
__device__ __forceinline__ void sgd_update(const DsgdArgs& a, float* prow, float* qrow, float* bup, float* bip,
                                           const float* isqp, float* cntp, float r, int gl, bool valid, int F4) {
    constexpr unsigned gmask = 0xFFFFFFFFu;  // callers keep whole warps converged (dummy ratings: valid == false)
    const int FP = F4 * 4;
    if (CH > 0) {
        constexpr int NCH = CH > 0 ? CH : 1;
        const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
        const bool tail_ok = gl + (NCH - 1) * G < F4;
        float4 p[NCH], q[NCH], z[NCH], g[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int ch = gl + c * G;
            const bool ok = (c + 1 < NCH) || tail_ok;
            p[c] = q[c] = z[c] = g[c] = zero4;
            if (ok) {
                p[c] = row_ld4<SU>(prow + 4 * ch);
                q[c] = row_ld4<SI>(qrow + 4 * ch);
                if (PP) {
                    z[c] = row_ld4<SU>(prow + FP + 4 * ch);
                    g[c] = row_ld4<SU>(prow + 2 * FP + 4 * ch);
                }
            }
        }
        float b_u = 0.f, b_i = 0.f, isq = 0.f, cnt = 0.f;
        if (BIASED) {
            b_u = sc_ld<SU>(bup);
            b_i = sc_ld<SI>(bip);
        }
        if (PP) {
            isq = sc_ld<SU>(isqp);
            cnt = sc_ld<SU>(cntp);
        }
        float part[NCH];
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            if (PP) { p[c].x += z[c].x; p[c].y += z[c].y; p[c].z += z[c].z; p[c].w += z[c].w; }  // p <- p + z
            part[c] = (p[c].x * q[c].x + p[c].y * q[c].y) + (p[c].z * q[c].z + p[c].w * q[c].w);
        }
        float dot = part[0];
        if (NCH == 2) dot = part[0] + part[1];
        if (NCH == 3) dot = (part[0] + part[1]) + part[2];
        if (NCH == 4) dot = (part[0] + part[1]) + (part[2] + part[3]);
        const float dp = 1.f - a.lr_pu * a.reg_pu, dq = 1.f - a.lr_qi * a.reg_qi, dy = 1.f - a.lr_yj * a.reg_yj;
        // The decayed old values (1 - lr reg) p, (1 - lr reg) q do not depend on the error: they are computed in
        // the shadow of the shuffle reduction (each stage is ~25 cycles during which this warp -- often the only
        // active one on its scheduler -- would issue nothing), so that only one FMA per element remains on the
        // critical path behind err.  Volatile asm keeps them between the shuffles where the source puts them.
        float4 pd[NCH], qd[NCH];
        auto scale4 = [](float4& o, float s, const float4& v) {
            asm volatile("mul.rn.f32 %0, %4, %5;\n\tmul.rn.f32 %1, %4, %6;\n\tmul.rn.f32 %2, %4, %7;\n\tmul.rn.f32 %3, %4, %8;"
                         : "=f"(o.x), "=f"(o.y), "=f"(o.z), "=f"(o.w)
                         : "f"(s), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
        };
        constexpr int NST = G >= 32 ? 5 : G >= 16 ? 4 : G >= 8 ? 3 : G >= 4 ? 2 : G >= 2 ? 1 : 0;  // shuffle stages
        int done = 0;  // float4 scale operations issued so far (2 per chunk)
        auto scale_some = [&](int upto) {
#pragma unroll
            for (int t = 0; t < 2 * NCH; ++t) {
                if (t >= done && t < upto) {
                    const int c = t >> 1;
                    if (t & 1) scale4(qd[c], dq, q[c]);
                    else {
                        float4 po = p[c];
                        if (PP) { po.x -= z[c].x; po.y -= z[c].y; po.z -= z[c].z; po.w -= z[c].w; }
                        scale4(pd[c], dp, po);
                    }
                }
            }
            done = upto > done ? upto : done;
        };
        const float mub = BIASED ? (a.mu + b_u) + b_i : 0.f;
        if (NST == 0) scale_some(2 * NCH);
        {
            int stage = 0;
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) {
                const float other = __shfl_xor_sync(gmask, dot, o);
                ++stage;
                scale_some((2 * NCH * stage + NST - 1) / NST);
                dot += other;
            }
        }
        const float err = BIASED ? r - (mub + dot) : r - dot;
        const float eg = err * isq;
        const float ep = a.lr_pu * err, eq = a.lr_qi * err, ey = a.lr_yj * err;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
            const int ch = gl + c * G;
            const bool st = valid && ((c + 1 < NCH) || tail_ok);
            const float4 pz = p[c];  // p (+ z for SVD++)
            // p + lr (err q - reg p) = (1 - lr reg) p + (lr err) q: one multiply (above) and one FMA per element
            float4 pn, qn;
            pn.x = fmaf(ep, q[c].x, pd[c].x);
            pn.y = fmaf(ep, q[c].y, pd[c].y);
            pn.z = fmaf(ep, q[c].z, pd[c].z);
            pn.w = fmaf(ep, q[c].w, pd[c].w);
            qn.x = fmaf(eq, pz.x, qd[c].x);
            qn.y = fmaf(eq, pz.y, qd[c].y);
            qn.z = fmaf(eq, pz.z, qd[c].z);
            qn.w = fmaf(eq, pz.w, qd[c].w);
            if (st) {
                row_st4<SU>(prow + 4 * ch, pn);
                row_st4<SI>(qrow + 4 * ch, qn);
            }
            if (PP) {
                float4 zn, gn;
                zn.x = fmaf(ey, q[c].x, dy * z[c].x);
                zn.y = fmaf(ey, q[c].y, dy * z[c].y);
                zn.z = fmaf(ey, q[c].z, dy * z[c].z);
                zn.w = fmaf(ey, q[c].w, dy * z[c].w);
                gn.x = g[c].x + eg * q[c].x; gn.y = g[c].y + eg * q[c].y;
                gn.z = g[c].z + eg * q[c].z; gn.w = g[c].w + eg * q[c].w;
                if (st) {
                    row_st4<SU>(prow + FP + 4 * ch, zn);
                    row_st4<SU>(prow + 2 * FP + 4 * ch, gn);
                }
            }
        }
        if (gl == 0 && valid) {
            if (BIASED) {
                sc_st<SU>(bup, b_u + a.lr_bu * (err - a.reg_bu * b_u));
                sc_st<SI>(bip, b_i + a.lr_bi * (err - a.reg_bi * b_i));
            }
            if (PP) sc_st<SU>(cntp, cnt + 1.f);
        }
        return;
    }
    float dot = 0.f;
    for (int c = gl; c < F4; c += G) {
        float4 p = row_ld4<SU>(prow + 4 * c);
        const float4 q = row_ld4<SI>(qrow + 4 * c);
        if (PP) {
            const float4 z = row_ld4<SU>(prow + FP + 4 * c);
            p.x += z.x; p.y += z.y; p.z += z.z; p.w += z.w;
        }
        dot += p.x * q.x + p.y * q.y + p.z * q.z + p.w * q.w;
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) dot += __shfl_xor_sync(gmask, dot, o);
    float err;
    if (BIASED) {
        const float b_u = sc_ld<SU>(bup), b_i = sc_ld<SI>(bip);
        err = r - (a.mu + b_u + b_i + dot);
        __syncwarp(gmask);  // every lane has read the biases before the leader overwrites them
        if (gl == 0 && valid) {
            sc_st<SU>(bup, b_u + a.lr_bu * (err - a.reg_bu * b_u));
            sc_st<SI>(bip, b_i + a.lr_bi * (err - a.reg_bi * b_i));
        }
    } else {
        err = r - dot;
    }
    float eg = 0.f;
    if (PP) {
        eg = err * sc_ld<SU>(isqp);
        const float cnt = sc_ld<SU>(cntp);
        __syncwarp(gmask);
        if (gl == 0 && valid) sc_st<SU>(cntp, cnt + 1.f);
    }
#pragma unroll 1
    for (int c = gl; c < F4 && valid; c += G) {
        const float4 p = row_ld4<SU>(prow + 4 * c), q = row_ld4<SI>(qrow + 4 * c);
        float4 pz = p, pn, qn;
        if (PP) {
            const float4 z = row_ld4<SU>(prow + FP + 4 * c), g = row_ld4<SU>(prow + 2 * FP + 4 * c);
            pz.x += z.x; pz.y += z.y; pz.z += z.z; pz.w += z.w;
            float4 zn, gn;
            zn.x = z.x + a.lr_yj * (err * q.x - a.reg_yj * z.x);
            zn.y = z.y + a.lr_yj * (err * q.y - a.reg_yj * z.y);
            zn.z = z.z + a.lr_yj * (err * q.z - a.reg_yj * z.z);
            zn.w = z.w + a.lr_yj * (err * q.w - a.reg_yj * z.w);
            gn.x = g.x + eg * q.x; gn.y = g.y + eg * q.y; gn.z = g.z + eg * q.z; gn.w = g.w + eg * q.w;
            row_st4<SU>(prow + FP + 4 * c, zn);
            row_st4<SU>(prow + 2 * FP + 4 * c, gn);
        }
        pn.x = p.x + a.lr_pu * (err * q.x - a.reg_pu * p.x);
        pn.y = p.y + a.lr_pu * (err * q.y - a.reg_pu * p.y);
        pn.z = p.z + a.lr_pu * (err * q.z - a.reg_pu * p.z);
        pn.w = p.w + a.lr_pu * (err * q.w - a.reg_pu * p.w);
        qn.x = q.x + a.lr_qi * (err * pz.x - a.reg_qi * q.x);
        qn.y = q.y + a.lr_qi * (err * pz.y - a.reg_qi * q.y);
        qn.z = q.z + a.lr_qi * (err * pz.z - a.reg_qi * q.z);
        qn.w = q.w + a.lr_qi * (err * pz.w - a.reg_qi * q.w);
        row_st4<SU>(prow + 4 * c, pn);
        row_st4<SI>(qrow + 4 * c, qn);
    }
}

// G lanes per rating, SU / SI: user / item block staged in shared memory, BIASED: SVD(biased=True)
// threads per CTA: 512 for G >= 16 (rows of 132..256 floats), else 256.  1024 threads would cap the kernel at 64
// registers, which the ring state alone nearly fills (spills).
__host__ __device__ constexpr int dsgd_threads(int g) { return g >= 16 ? 512 : 256; }

// DEP (G = 32: one warp per rating): instead of waves separated by block barriers, every warp walks its share of the
// cell's records (record k -> warp k % n_warps, records in colour order) and starts a rating as soon as the two
// rows it touches carry exactly the updates that precede it in that order -- per-row version counters in shared
// memory, ld.acquire / st.release at CTA scope.  Same conflict-freedom and determinism as the waves (every row sees
// its updates in the same fixed order), but a cell costs its dependency chain (max degree x one update latency)
// or its work / n_warps, whichever is longer, not (number of waves) x (slowest warp of the wave + barrier).
template <int G, int CH, bool SU, bool SI, bool BIASED, bool PP, bool DEP = false>
__device__ __forceinline__ void dsgd_body(const DsgdArgs& a, const int ub) {
    extern __shared__ __align__(16) float smem_f[];
    const int B = a.B, W = a.W, FP = a.FP, F4 = a.FP >> 2;
    const int US = a.US, U4 = a.US >> 2;  // user rows: US floats ([p] or [p | z | g])
    const int tid = threadIdx.x, nthr = blockDim.x;
    const int gid = tid / G, gl = tid % G;
    const int gid0 = (tid & ~31) / G;  // first lane-group of this warp

    // shared memory carve-up
    // item-block buffers: [max_il x FP factors | max_il biases], two of them when blocks hop through DSMEM
    float* pu_s = smem_f;
    float* ibuf_s = pu_s + (SU ? (size_t)a.max_ul * US : 0);
    float* bu_s = ibuf_s + (SI ? (size_t)(a.C > 1 ? 2 : 1) * a.ibuf : 0);
    float* isq_s = bu_s + (SU ? a.max_ul : 0);
    float* cnt_s = isq_s + ((SU && PP) ? a.max_ul : 0);
    int* wave_s = reinterpret_cast<int*>(cnt_s + ((SU && PP) ? a.max_ul : 0));
    int* coff_s = wave_s + 2 * (NW + 1);      // [2 * P * B]: cell begin / end per stratum (wave_s: two buffers)
    int* rul_s = coff_s + 2 * a.P * B;        // records: two buffers of rec_cap each
    int* ril_s = rul_s + 2 * a.rec_cap;
    float* rr_s = reinterpret_cast<float*>(ril_s + 2 * a.rec_cap);
    int* rdep_s = reinterpret_cast<int*>(rr_s + 2 * a.rec_cap);   // DEP: two buffers of rec_cap
    int* ver_s = rdep_s + (DEP ? 2 * a.rec_cap : 0);              // DEP: [max_ul] user-row + [max_il] item-row versions

    // ring mailboxes (clusters): bar_data = "my right neighbour's push has landed in my spare buffer",
    // bar_free = "my left neighbour has finished reading the buffer I am about to overwrite"
    // Two of each, used alternately (push number & 1): a neighbour can run one push ahead of the CTA that waits,
    // and a single mbarrier cannot tell "one phase ahead" from "not yet" once two phases have completed.
    __shared__ __align__(8) uint64_t ring_bar[4];  // [0,1] data, [2,3] free
    if (tid == 0) {
        // per-lane hop: one arrival per warp; bulk hop: one arrival per mailbox phase (see the hop below)
        for (int x = 0; x < 4; ++x) mbar_init_cta(&ring_bar[x], a.bulk_hop ? 1u : (uint32_t)(nthr >> 5));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const int nu_local = (a.n_users - ub + B - 1) / B;
    if (SU) {
        for (int l = tid / U4, c = tid % U4; l < nu_local; ) {
            reinterpret_cast<float4*>(pu_s)[l * U4 + c] =
                __ldcg(reinterpret_cast<const float4*>(a.pu + ((size_t)(ub + (size_t)l * B)) * US) + c);
            c += nthr % U4; l += nthr / U4;
            if (c >= U4) { c -= U4; ++l; }
        }
        for (int l = tid; l < nu_local; l += nthr) {
            bu_s[l] = __ldcg(a.bu + ub + (size_t)l * B);
            if (PP) {
                isq_s[l] = __ldcg(a.isq + ub + (size_t)l * B);
                cnt_s[l] = __ldcg(a.cnt + ub + (size_t)l * B);
            }
        }
    }
    for (int s = tid; s < a.P * B; s += nthr) {
        coff_s[2 * s] = a.cell_off[(size_t)s * B + ub];
        coff_s[2 * s + 1] = a.cell_off[(size_t)s * B + ub + 1];
    }
    __syncthreads();
    SpinGuard guard{a.status, false};

    long long t_wait = 0, t_load = 0, t_upd = 0, t_wb = 0, n_wave = 0, t_hop = 0, t_free = 0, t_push = 0;
#ifdef SB2_DSGD_CHECK
    // debug build (-DSB2_DSGD_CHECK): every rating of a wave stamps its user row and its item row with the wave's
    // number; a row that already carries the stamp is shared by two ratings of one wave -- a schedule conflict,
    // reported through status[3] (sb2_svd_plan_status fails).  Rows beyond CHK_ROWS per block are not checked.
    constexpr int CHK_ROWS = 2048;
    __shared__ int chk_u[CHK_ROWS], chk_i[CHK_ROWS];
    for (int x = tid; x < CHK_ROWS; x += nthr) { chk_u[x] = 0; chk_i[x] = 0; }
    __syncthreads();
    auto stamp = [&](int ul, int il, bool valid, int tag) {
        if (valid && gl == 0) {
            if (ul < CHK_ROWS && atomicExch(&chk_u[ul], tag) == tag) atomicOr(&a.status[3], 1);
            if (il < CHK_ROWS && atomicExch(&chk_i[il], tag) == tag) atomicOr(&a.status[3], 2);
            atomicAdd(&a.status[2], 1);   // ratings checked
        }
    };
#endif
#ifdef SB2_DSGD_WAVE_PROF
    long long t_act = 0, t_bar = 0;  // warp 0: cycles inside the updates of a wave / in the barrier after it
#endif
    // Two-level ring.  CTAs form clusters of C; cluster Cl owns user blocks Cl*C .. Cl*C+C-1.  Item blocks form
    // K = B / C super-blocks of C blocks.  Outer step T: super-block D = (Cl + T) % K is resident in the
    // cluster; inner step t: CTA c updates item block (D, (c + t) % C) and then pushes it into its left
    // neighbour's spare buffer through distributed shared memory (two cluster barriers, no global traffic).
    // Only the K hand-offs between clusters go through L2 with the release / acquire step counters.
    const int C = a.C, K = B / C;
    const int Cl = ub / C, c = ub - Cl * C;
    // a launch covers strata [s_begin, s_end) (s = T * C + t); it may start and end in the middle of an outer step
    // (SVD++ chunks): the first stratum of a launch always loads its block from global memory (everything was
    // written back when the previous launch ended) and the last one always writes back.
    const int T_begin = a.s_begin / C, T_end = (a.s_end + C - 1) / C;
    const int n_outer = T_end - T_begin;
    int slot = 0;
    uint32_t n_push = 0;  // pushes done so far (selects the mbarrier phases)
    uint32_t left_data_bar = 0, right_free_bar = 0;  // remote addresses of ring_bar[0] (left) / ring_bar[2] (right)
    uint32_t right2_free_bar = 0;                    // ring_bar[2] of the CTA two to the right (bulk hop)
    if (C > 1) {
        cluster_sync_all();  // every CTA's mailboxes are initialised before anybody arrives on them
        left_data_bar = dsmem_addr(&ring_bar[0], (uint32_t)(c == 0 ? C - 1 : c - 1));
        right_free_bar = dsmem_addr(&ring_bar[2], (uint32_t)(c + 1 == C ? 0 : c + 1));
        right2_free_bar = dsmem_addr(&ring_bar[2], (uint32_t)((c + 2) % C));
    }
    const int n_strata = a.s_end - a.s_begin;
    const int n_steps = a.n_epochs * n_strata;
    // records + wave table of step j go to buffer (j & 1) with cp.async, issued one step ahead: they land while
    // the previous stratum is being updated instead of costing an L2 round trip at the head of every stratum
    auto prefetch = [&](int j, int s) {   // step j works on stratum s of the epoch, s in [0, P * B)
        const int k0 = coff_s[2 * s];
        const int staged = min(coff_s[2 * s + 1] - k0, a.rec_cap);
        int* rul = rul_s + (size_t)(j & 1) * a.rec_cap;
        int* ril = ril_s + (size_t)(j & 1) * a.rec_cap;
        float* rr = rr_s + (size_t)(j & 1) * a.rec_cap;
        int* wave = wave_s + (j & 1) * (NW + 1);
        for (int x = tid; x < staged; x += nthr) {
            cp_async4(rul + x, a.ul + k0 + x);
            cp_async4(ril + x, a.il + k0 + x);
            cp_async4(rr + x, a.r + k0 + x);
            if (DEP) cp_async4(rdep_s + (size_t)(j & 1) * a.rec_cap + x, a.dep + k0 + x);
        }
        if (!DEP) {
            const int* wsrc = a.wave_off + ((size_t)s * B + ub) * (NW + 1);
            for (int x = tid; x <= NW; x += nthr) cp_async4(wave + x, wsrc + x);
        }
    };
    if (n_steps > 0) prefetch(0, a.s_begin);
    const int P = a.P;
    // position of the current step, advanced incrementally at the bottom of the loop (a handful of integer divisions
    // per stratum are ~0.3k cycles of a 9k-cycle stratum): epoch ep, stratum sg of the epoch, sub-epoch S and local
    // stratum s (ranks), outer / inner step (T, t), resident super-block D = (Cl + T) % K
    const int ni_q = a.n_items / B, ni_r = a.n_items - ni_q * B;   // items of block ib (one rank): ni_q + (ib < ni_r)
    int ep = 0, sg = a.s_begin;
    int S = P > 1 ? sg / B : 0;
    int s = sg - S * B;
    int T = s / C, t = s - T * C;
    int D = (Cl + T) % K;
    for (int step = 0; step < n_steps; ++step) {
        // ranks: E sub-epochs since the fit began; launches of a ring cover whole epochs
        const int E = a.E_base + ep * P + S;
        const int gstep = P > 1 ? E * K + T : ep * n_outer + (T - T_begin);
        const bool first = (sg == a.s_begin) || t == 0;       // of this outer step within the launch
        const bool last = (sg + 1 == a.s_end) || t + 1 == C;
        const bool wait_flag = P > 1 ? (first && gstep != 0) : (first && step != 0);
        // where this sub-epoch's item rows live in global memory (the L2 hand-off between clusters, block loads)
        float* g_qi = a.qi;
        float* g_bi = a.bi;
        int n_items_sb = a.n_items;
        if (P > 1) {
            g_qi = a.ring_qi[E & 1];
            g_bi = a.ring_bi[E & 1];
            int sb = (a.rank + E) % P;
            n_items_sb = (a.n_items_glob - sb + P - 1) / P;
        }
        const int* rul_c = rul_s + (size_t)(step & 1) * a.rec_cap;
        const int* ril_c = ril_s + (size_t)(step & 1) * a.rec_cap;
        const float* rr_c = rr_s + (size_t)(step & 1) * a.rec_cap;
        const int* wave_c = wave_s + (step & 1) * (NW + 1);
        int j = c + t;
        if (j >= C) j -= C;
        const int ib = D * C + j;
        float* qi_s = ibuf_s + (size_t)slot * a.ibuf;
        float* bi_s = qi_s + (size_t)a.max_il * FP;
        const long long c0 = clock64();
        // a wait that ran into its deadline anywhere (on this GPU) ends all mailbox traffic of the draining launch:
        // the word is read here and looked at at the hop, a stratum later
        const int status_now = ld_relaxed(a.status);
        const int k0 = coff_s[2 * sg], cnt = coff_s[2 * sg + 1] - k0;
        const int staged = min(cnt, a.rec_cap);
        cp_async_wait_all();  // this stratum's records (issued during the previous stratum)
        if (DEP)
            for (int x = tid; x < a.max_ul + a.max_il; x += nthr) ver_s[x] = 0;
        if (wait_flag && tid == 0) {
            // T > 0 (or one rank): the previous cluster still owns the block; T == 0 of a ring: the right
            // neighbour rank delivers it at the end of ITS previous sub-epoch (system-scope release over NVLink)
            if (P > 1 && T == 0) wait_counter<WAIT_GE_SYS>(guard, a.rflags + ib, E);
            else wait_counter<WAIT_EQ_GPU>(guard, a.flags + ib, gstep);
        }
        __syncthreads();
        if (step + 1 < n_steps) prefetch(step + 1, sg + 1 == a.s_end ? a.s_begin : sg + 1);
        const long long c1 = clock64();
        const int ni_local = P > 1 ? (n_items_sb - ib + B - 1) / B : ni_q + (ib < ni_r ? 1 : 0);
        if (SI && first) {
            const int total = ni_local * F4;
            for (int t0 = tid; t0 < total; t0 += 4 * nthr) {
                float4 v[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int x = t0 + q * nthr;
                    if (x < total) {
                        const int l = x / F4, cc = x - l * F4;
                        v[q] = __ldcg(reinterpret_cast<const float4*>(g_qi + ((size_t)(ib + (size_t)l * B)) * FP) + cc);
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int x = t0 + q * nthr;
                    if (x < total) reinterpret_cast<float4*>(qi_s)[x] = v[q];
                }
            }
            for (int l = tid; l < ni_local; l += nthr) bi_s[l] = __ldcg(g_bi + ib + (size_t)l * B);
            __syncthreads();
            // ring: this was the last read of slot ib of buffer E & 1 in this sub-epoch (the block leaves the rank
            // at the end of the outer step): the right neighbour may overwrite it with the block of sub-epoch E + 2
            if (P > 1 && T == K - 1 && tid == 0) st_release_sys(a.right_credit + ib, E + 1);
        }
        const long long c2 = clock64();

        // every lane-group runs the same (CTA-uniform) number of rounds per wave, groups beyond the wave's
        // end carry a dummy rating with all stores predicated off: control flow stays warp-uniform, so the
        // shuffles can use the full-warp mask (a per-group mask costs MATCH / VOTE instructions per shuffle)
        // the record of a rating: fetched one wave ahead (shared-memory reads of read-only data), so that the wave's
        // critical path starts at the row loads instead of at wave table -> record -> address
        auto fetch = [&](int k, bool valid, int& ul, int& il, float& r) {
            ul = 0; il = 0; r = 0.f;
            if (valid) {
                if (k < staged) { ul = rul_c[k]; il = ril_c[k]; r = rr_c[k]; }
                else { ul = a.ul[k0 + k]; il = a.il[k0 + k]; r = a.r[k0 + k]; }
            }
        };
        auto update = [&](int ul, int il, float r, bool valid) {
            float* prow = SU ? pu_s + (size_t)ul * US : a.pu + ((size_t)(ub + (size_t)ul * B)) * US;
            float* qrow = SI ? qi_s + (size_t)il * FP : g_qi + ((size_t)(ib + (size_t)il * B)) * FP;
            float* bup = SU ? bu_s + ul : a.bu + ub + (size_t)ul * B;
            float* bip = SI ? bi_s + il : g_bi + ib + (size_t)il * B;
            const float* isqp = PP ? (SU ? isq_s + ul : a.isq + ub + (size_t)ul * B) : nullptr;
            float* cntp = PP ? (SU ? cnt_s + ul : a.cnt + ub + (size_t)ul * B) : nullptr;
            sgd_update<G, CH, SU, SI, BIASED, PP>(a, prow, qrow, bup, bip, isqp, cntp, r, gl, valid, F4);
        };
        auto process = [&](int k, bool valid) {
            int ul, il;
            float r;
            fetch(k, valid, ul, il, r);
            update(ul, il, r, valid);
        };
        if (DEP) {
            const int* rdep_c = rdep_s + (size_t)(step & 1) * a.rec_cap;
            int* ver_u = ver_s;
            int* ver_i = ver_s + a.max_ul;
            for (int k = gid; k < cnt; k += W) {   // G == 32: gid = warp, W = warps
                int ul, il, dep;
                float r;
                if (k < staged) { ul = rul_c[k]; il = ril_c[k]; r = rr_c[k]; dep = rdep_c[k]; }
                else { ul = a.ul[k0 + k]; il = a.il[k0 + k]; r = a.r[k0 + k]; dep = a.dep[k0 + k]; }
                const int nu = dep & 0xFFFF, nv = (dep >> 16) & 0xFFFF;
                // both rows must carry exactly the updates that precede this rating in the cell's order (every lane
                // acquires for itself; the addresses are warp-uniform: broadcast reads).  The producers are warps of
                // this CTA working through earlier records: the earliest unfinished record never waits.
                while (ld_acquire_cta_shared(ver_u + ul) != nu || ld_acquire_cta_shared(ver_i + il) != nv) { }
                update(ul, il, r, true);
                __syncwarp();  // orders the lanes' row stores before lane 0's releases
                if (gl == 0) {
                    if (a.dep_sync == 0) {
                        st_release_cta_shared(ver_u + ul, nu + 1);
                        st_release_cta_shared(ver_i + il, nv + 1);
                    } else {
                        if (a.dep_sync == 1) asm volatile("fence.acq_rel.cta;" ::: "memory");
                        *reinterpret_cast<volatile int*>(ver_u + ul) = nu + 1;
                        *reinterpret_cast<volatile int*>(ver_i + il) = nv + 1;
                    }
                }
                ++n_wave;
            }
            __syncthreads();
        } else {
        {
            int wb = wave_c[0], we = wave_c[1];
            int c_ul, c_il;
            float c_r;
            fetch(wb + gid, wb + gid < we, c_ul, c_il, c_r);
            for (int w = 0; w < NW - 1; ++w) {
                if (wb == we) break;  // colours are contiguous: an empty wave ends the cell (CTA-uniform)
                // first round of the NEXT wave (wave NW - 1 is the tail: fetched and ignored)
                const int nwb = we, nwe = wave_c[w + 2];
                int n_ul, n_il;
                float n_r;
                fetch(nwb + gid, w + 2 < NW && nwb + gid < nwe, n_ul, n_il, n_r);
#ifdef SB2_DSGD_WAVE_PROF
                const long long w0 = clock64();
#endif
                // a warp whose first lane-group is already past the wave's end holds only dummies: skip it
                // (warp-uniform test), it would otherwise compete for issue slots with the working warps
#ifdef SB2_DSGD_CHECK
                {
                    const int tag = step * NW + w + 1;
                    stamp(c_ul, c_il, wb + gid < we, tag);
                    for (int k = wb + W; k < we; k += W) {
                        int x_ul, x_il;
                        float x_r;
                        fetch(k + gid, k + gid < we, x_ul, x_il, x_r);
                        stamp(x_ul, x_il, k + gid < we, tag);
                    }
                }
#endif
                if (wb + gid0 < we) update(c_ul, c_il, c_r, wb + gid < we);
                for (int k = wb + W; k < we; k += W)
                    if (k + gid0 < we) process(k + gid, k + gid < we);
                ++n_wave;
#ifdef SB2_DSGD_WAVE_PROF
                const long long w1 = clock64();
                __syncthreads();
                t_act += w1 - w0;
                t_bar += clock64() - w1;
#else
                __syncthreads();
#endif
                wb = nwb; we = nwe; c_ul = n_ul; c_il = n_il; c_r = n_r;
            }
        }
        {
            const int wb = wave_c[NW - 1], we = wave_c[NW];
            if (wb != we) {  // sequential tail (colour overflow), the first warp replays it in order
                if (tid < 32)
                    for (int k = wb; k < we; ++k) {
                        process(k, gid == 0);
                        __syncwarp();  // consecutive tail ratings may share a row
                    }
                __syncthreads();
            }
        }
        }
        const long long c3 = clock64();
        if (!last && a.bulk_hop) {
            // fast hop, asynchronous: ONE thread hands the block (a.ibuf floats) to the copy engine, which writes it into
            // the left neighbour's spare buffer and completes the bytes on the neighbour's data mailbox; no lane
            // stores, no cluster-scope fence.
            //   data mailbox  D[k & 1] of push k: this CTA's own arrive.expect_tx + the bytes of the incoming copy
            //   free mailbox  F[k & 1]: CTA x, once push k has landed in its buffer (so the sender x + 1 no longer needs
            //     its source buffer), arrives on F[k & 1] of CTA x + 2, the one that writes into x + 1's buffers:
            //     push k + 1 of x + 2 may overwrite that source.  The arrival publishes no data of this CTA (the copy
            //     engine's reads of the source are over when its bytes have landed): relaxed, and the waits are
            //     CTA-scope -- a release / acquire pair at cluster scope costs a MEMBAR.ALL.GPU and an L1 invalidation
            //     per stratum on the path of the thread every other warp then waits for.
            // The source buffer is only read by the copy engine, the working buffer only by this CTA's threads, and a
            // mailbox is reused every second push, which the free mailbox orders behind the previous use.
            fence_proxy_async_smem();
            __syncthreads();
            const long long c4 = clock64();
            if (status_now != 0) guard.dead = true;
            if (tid == 0) {
                if (n_push > 0) mbar_wait_cta(guard, &ring_bar[2 + ((n_push - 1) & 1)], ((n_push - 1) >> 1) & 1);
                const uint32_t bytes = (uint32_t)a.ibuf * 4u;
                const uint32_t dst = dsmem_addr(ibuf_s + (size_t)(slot ^ 1) * a.ibuf, (uint32_t)(c == 0 ? C - 1 : c - 1));
                if (!guard.dead) {   // a draining launch posts nothing: no transaction count may pile up on a mailbox
                    mbar_arrive_expect_tx(&ring_bar[n_push & 1], bytes);
                    dsmem_bulk_push(dst, qi_s, bytes, left_data_bar + 8u * (n_push & 1));
                }
            }
            const long long c5 = clock64();
            mbar_wait_cta(guard, &ring_bar[n_push & 1], (n_push >> 1) & 1);
            if (tid == 0 && !guard.dead) mbar_arrive_remote_relaxed(right2_free_bar + 8u * (n_push & 1));
            ++n_push;
            slot ^= 1;
            t_free += c4 - c3; t_push += c5 - c4;
            t_hop += clock64() - c3;
        } else if (!last) {
            // fast hop (neighbour-to-neighbour, no cluster-wide barrier): once the left neighbour has finished
            // reading its spare buffer (its previous push), copy my block into it through distributed shared
            // memory, tell it the data is there, tell my right neighbour that my block buffer is reusable,
            // and wait for my right neighbour's push into my own spare buffer.
            // Every thread waits for "free" itself and every warp signals for itself (mailboxes count one arrival
            // per warp): no block barrier and no single-thread relay inside the hop.  __syncwarp orders the lanes'
            // remote stores (and their reads of the block being sent) before lane 0's cluster-scope releases.
            if (n_push > 0) mbar_wait_cluster(guard, &ring_bar[2 + ((n_push - 1) & 1)], ((n_push - 1) >> 1) & 1);
            const long long c4 = clock64();
            const uint32_t dst = dsmem_addr(ibuf_s + (size_t)(slot ^ 1) * a.ibuf, (uint32_t)(c == 0 ? C - 1 : c - 1));
            const int n4 = a.ibuf >> 2;
            for (int x = tid; x < n4; x += nthr) dsmem_st4(dst + 16u * x, reinterpret_cast<const float4*>(qi_s)[x]);
            __syncwarp();
            if ((tid & 31) == 0) {
                asm volatile("fence.acq_rel.cluster;" ::: "memory");
                mbar_arrive_remote_relaxed(left_data_bar + 8u * (n_push & 1));
                mbar_arrive_remote_relaxed(right_free_bar + 8u * (n_push & 1));
            }
            const long long c5 = clock64();
            t_free += c4 - c3; t_push += c5 - c4;
            mbar_wait_cluster(guard, &ring_bar[n_push & 1], (n_push >> 1) & 1);
            ++n_push;
            slot ^= 1;
            t_hop += clock64() - c3;
        } else {
            // slow hop: hand the block to the next cluster through L2 -- or, at the end of a ring's sub-epoch, to
            // the left neighbour RANK: the rows are stored straight into its buffer (E + 1) & 1 through the
            // peer mapping (NVLink), once it has returned the credit for that slot
            float* d_qi = g_qi;
            float* d_bi = g_bi;
            const bool to_peer = P > 1 && T == K - 1;
            if (to_peer) {
                d_qi = a.left_qi[(E + 1) & 1];
                d_bi = a.left_bi[(E + 1) & 1];
                if (tid == 0) wait_counter<WAIT_GE_SYS>(guard, a.credit + ib, E);
                __syncthreads();
            }
            if (SI) {
                for (int l = tid / F4, cc = tid % F4; l < ni_local; ) {
                    __stcg(reinterpret_cast<float4*>(d_qi + ((size_t)(ib + (size_t)l * B)) * FP) + cc,
                           reinterpret_cast<const float4*>(qi_s)[l * F4 + cc]);
                    cc += nthr % F4; l += nthr / F4;
                    if (cc >= F4) { cc -= F4; ++l; }
                }
                if (BIASED)
                    for (int l = tid; l < ni_local; l += nthr) __stcg(d_bi + ib + (size_t)l * B, bi_s[l]);
            }
            // bar.sync orders every thread's stores before thread 0's release (cumulativity); system scope when
            // the consumer is another GPU
            __syncthreads();
            if (tid == 0) {
                if (to_peer) st_release_sys(a.left_rflags + ib, E + 1);
                else st_release(a.flags + ib, gstep + 1);
            }
            t_wb += clock64() - c3;
        }
        t_wait += c1 - c0; t_load += c2 - c1; t_upd += c3 - c2;
        // advance to the next stratum
        ++sg; ++s; ++t;
        if (t == C) { t = 0; ++T; D = D + 1 == K ? 0 : D + 1; }
        if (sg == a.s_end) {            // next epoch of this launch
            sg = a.s_begin; ++ep;
            S = P > 1 ? sg / B : 0; s = sg - S * B; T = s / C; t = s - T * C; D = (Cl + T) % K;
        } else if (s == B) {            // next sub-epoch (rings only: one rank has s_end <= B)
            s = 0; ++S; T = 0; t = 0; D = Cl % K;
        }
    }
    if (C > 1) cluster_sync_all();  // no CTA leaves while a neighbour may still address its shared memory
    if (a.prof != nullptr && tid == 0) {
        a.prof[ub * 8 + 0] = t_wait; a.prof[ub * 8 + 1] = t_load; a.prof[ub * 8 + 2] = t_upd; a.prof[ub * 8 + 3] = t_wb;
        a.prof[ub * 8 + 4] = t_free; a.prof[ub * 8 + 5] = t_push; a.prof[ub * 8 + 6] = n_wave; a.prof[ub * 8 + 7] = t_hop;
#ifdef SB2_DSGD_WAVE_PROF
        a.prof[ub * 8 + 4] = t_act; a.prof[ub * 8 + 5] = t_bar;
#endif
    }
    if (SU) {
        for (int l = tid / U4, c = tid % U4; l < nu_local; ) {
            __stcg(reinterpret_cast<float4*>(a.pu + ((size_t)(ub + (size_t)l * B)) * US) + c,
                   reinterpret_cast<const float4*>(pu_s)[l * U4 + c]);
            c += nthr % U4; l += nthr / U4;
            if (c >= U4) { c -= U4; ++l; }
        }
        for (int l = tid; l < nu_local; l += nthr) {
            if (BIASED) __stcg(a.bu + ub + (size_t)l * B, bu_s[l]);
            if (PP) __stcg(a.cnt + ub + (size_t)l * B, cnt_s[l]);
        }
    }
}

template <int G, int CH, bool SU, bool SI, bool BIASED, bool PP, bool DEP = false>
__global__ void __launch_bounds__(dsgd_threads(G), 1) dsgd_svd_kernel(const DsgdArgs a) {
    dsgd_body<G, CH, SU, SI, BIASED, PP, DEP>(a, blockIdx.x);
}

// All ranks of a ring in ONE launch (tests on a single GPU): the grid is n x B CTAs, CTA b works as CTA b % B of
// rank b / B with that rank's arguments -- exactly the code of a real rank, the "peer" buffers simply being the other
// ranks' slabs in the same memory.  Kernels that wait for each other must not be issued as separate launches on one
// GPU (nothing guarantees that they run at the same time); one launch whose CTAs are all resident does.  B is a
// multiple of the cluster size, so clusters never straddle ranks.
constexpr int DSGD_MAX_VIRTUAL = 4;
struct DsgdMulti {
    DsgdArgs r[DSGD_MAX_VIRTUAL];
};
template <int G, int CH, bool BIASED, bool PP>
__global__ void __launch_bounds__(dsgd_threads(G), 1) dsgd_svd_multi_kernel(const DsgdMulti m) {
    const int B = m.r[0].B;
    const int rank = blockIdx.x / B;
    dsgd_body<G, CH, true, true, BIASED, PP, false>(m.r[rank], blockIdx.x - rank * B);
}

// ------------------------------------------------------------------------------------------------
// preparation kernels: cell key -> stable sort -> per-cell greedy edge colouring -> wave tables
// ------------------------------------------------------------------------------------------------
__global__ void dsgd_key_kernel(int64_t n, const int32_t* __restrict__ u, const int32_t* __restrict__ i, int B, int C,
                                int P, int rank, int n_users, int n_items, unsigned n_cells, unsigned* __restrict__ key,
                                int* __restrict__ val, int* __restrict__ cnt, int* status) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int uu = u[k], ii = i[k];
    val[k] = (int)k;
    if (uu < 0 || uu >= n_users || ii < 0 || ii >= n_items) {
        atomicExch(status, 1);
        key[k] = n_cells;
        return;
    }
    // ring over P ranks: this rank keeps the ratings of its own users (u % P == rank); the others sort behind
    // the last cell.  Local ids: user u / P, item i / P inside super-block i % P, visited in sub-epoch S.
    if (uu % P != rank) {
        key[k] = n_cells;
        return;
    }
    const int S = ((ii % P) - rank + P) % P;
    const int ub = (uu / P) % B, ibk = (ii / P) % B;
    // stratum of the two-level ring: outer step T moves super-blocks between clusters, inner step t inside
    const int K = B / C;
    const int Cl = ub / C, c = ub % C, D = ibk / C, j = ibk % C;
    const int T = (D - Cl + K) % K, t = (j - c + C) % C;
    const int s = S * B + T * C + t;
    const unsigned cell = (unsigned)(s * B + ub);
    key[k] = cell;
    atomicAdd(&cnt[cell], 1);
}

// One warp per cell.  Lane 0 walks the cell's ratings in their (stable) input order and gives each the
// lowest colour not yet used by its user or its item (64-bit masks in shared memory); colours >= 63
// share the sequential tail.  Then a counting sort by colour writes the records and the wave table, and
// (dep_out != nullptr) each record's dependency counts for the DEP kernels: the number of records on the same
// user row / item row that precede it in the colour-sorted order.  A proper colour occurs at most once per row, so
// that is a popcount of the row's final mask below the record's colour; tail records (several per row possible)
// follow all coloured ones in placement order.
constexpr int COLOR_CAP = 512;  // ratings of a cell staged in shared memory at a time
__global__ void __launch_bounds__(32) dsgd_color_kernel(int n_cells, int B, int P, int max_ul, int max_il,
                                                        const int* __restrict__ cell_off, const int* __restrict__ val,
                                                        const int32_t* __restrict__ u, const int32_t* __restrict__ i,
                                                        const double* __restrict__ r, uint8_t* __restrict__ color_tmp,
                                                        int* __restrict__ ul_out, int* __restrict__ il_out,
                                                        float* __restrict__ r_out, int* __restrict__ wave_off,
                                                        int* __restrict__ dep_out, int* status) {
    extern __shared__ unsigned long long masks[];  // [max_ul] user masks, [max_il] item masks, then int tail counters
    int* tail_cnt = reinterpret_cast<int*>(masks + max_ul + max_il);
    __shared__ int hist[NW + 1];
    // the greedy colouring is sequential (lane 0), everything around it is not: the 32 lanes fetch a chunk of the
    // cell's ratings (three dependent global reads each: position -> (u, i) -> local rows) into shared memory, lane 0
    // colours / places the chunk out of shared memory, the 32 lanes write the results
    __shared__ int s_src[COLOR_CAP], s_ul[COLOR_CAP], s_il[COLOR_CAP], s_pos[COLOR_CAP], s_dep[COLOR_CAP];
    __shared__ uint8_t s_col[COLOR_CAP];
    const int lane = threadIdx.x;
    for (int cell = blockIdx.x; cell < n_cells; cell += gridDim.x) {
        const int k0 = cell_off[cell], k1 = cell_off[cell + 1];
        for (int t = lane; t < max_ul + max_il; t += 32) { masks[t] = 0ull; tail_cnt[t] = 0; }
        for (int t = lane; t <= NW; t += 32) hist[t] = 0;
        if (lane == 0) atomicMax(&status[1], k1 - k0);
        __syncwarp();
        auto stage = [&](int c0, int n, bool with_colour) {
            for (int t = lane; t < n; t += 32) {
                const int src = val[c0 + t];
                s_src[t] = src;
                s_ul[t] = (u[src] / P) / B;
                s_il[t] = (i[src] / P) / B;
                if (with_colour) s_col[t] = color_tmp[c0 + t];
            }
            __syncwarp();
        };
        // pass 1: colours in the cell's (stable) input order
        for (int c0 = k0; c0 < k1; c0 += COLOR_CAP) {
            const int n = min(COLOR_CAP, k1 - c0);
            stage(c0, n, false);
            if (lane == 0) {
                for (int t = 0; t < n; ++t) {
                    const int ul = s_ul[t], il = s_il[t];
                    const unsigned long long used = masks[ul] | masks[max_ul + il];
                    int c = __ffsll((long long)~used) - 1;  // lowest free colour, -1 if none
                    if (c < 0 || c >= NW - 1) c = NW - 1;
                    else {
                        masks[ul] |= 1ull << c;
                        masks[max_ul + il] |= 1ull << c;
                    }
                    s_col[t] = (uint8_t)c;
                    hist[c + 1]++;
                }
            }
            __syncwarp();
            if (k1 - k0 > COLOR_CAP)   // a single chunk stays in shared memory for pass 2
                for (int t = lane; t < n; t += 32) color_tmp[c0 + t] = s_col[t];
            __syncwarp();
        }
        if (lane == 0)
            for (int c = 0; c < NW; ++c) hist[c + 1] += hist[c];
        __syncwarp();
        for (int c = lane; c <= NW; c += 32) wave_off[(size_t)cell * (NW + 1) + c] = hist[c];
        __syncwarp();
        // pass 2: counting sort by colour (stable), dependency counts for the DEP kernels
        int worst = 0;
        for (int c0 = k0; c0 < k1; c0 += COLOR_CAP) {
            const int n = min(COLOR_CAP, k1 - c0);
            if (k1 - k0 > COLOR_CAP) stage(c0, n, true);
            if (lane == 0) {
                for (int t = 0; t < n; ++t) {
                    const int c = s_col[t];
                    s_pos[t] = k0 + hist[c]++;
                    if (dep_out != nullptr) {
                        const int ul = s_ul[t], il = s_il[t];
                        int nu, nv;
                        if (c < NW - 1) {
                            const unsigned long long below = (1ull << c) - 1ull;
                            nu = __popcll(masks[ul] & below);
                            nv = __popcll(masks[max_ul + il] & below);
                        } else {
                            nu = __popcll(masks[ul]) + tail_cnt[ul]++;
                            nv = __popcll(masks[max_ul + il]) + tail_cnt[max_ul + il]++;
                        }
                        worst = max(worst, max(nu, nv));
                        s_dep[t] = (nu & 0xFFFF) | (nv << 16);
                    }
                }
            }
            __syncwarp();
            for (int t = lane; t < n; t += 32) {
                const int pos = s_pos[t];
                ul_out[pos] = s_ul[t];
                il_out[pos] = s_il[t];
                r_out[pos] = (float)r[s_src[t]];
                if (dep_out != nullptr) dep_out[pos] = s_dep[t];
            }
            __syncwarp();
        }
        if (dep_out != nullptr && lane == 0) atomicMax(&status[2], worst);
        __syncwarp();
    }
}

// fp64 (rows x f) -> fp32 rows of `stride` floats: [0, f) = src, [f, stride) = 0; local row l <- source row
// first + l * step (ring: the rows of one rank / super-block)
__global__ void f64_to_rows_kernel(int64_t rows, int f, int stride, const double* __restrict__ src, float* __restrict__ dst,
                                   int64_t first, int64_t step) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= rows * stride) return;
    const int64_t row = t / stride;
    const int c = (int)(t % stride);
    dst[t] = c < f ? (float)src[(first + row * step) * f + c] : 0.f;
}

// ---- SVD++ companions of the stratified kernel --------------------------------------------------
// z_u = sum_{j in I_u} y_j / sqrt|I_u|  (matrix_factorization.pyx:472-476), and reset of g_u / cnt_u.
// One warp per user; user rows are [p | z | g] with stride US = 3 * FP.
__global__ void svdpp_user_refresh_kernel(int64_t n_users, int FP, const int64_t* __restrict__ u_ptr,
                                          const int32_t* __restrict__ ui_idx, const float* __restrict__ yj,
                                          const float* __restrict__ isq, float* __restrict__ urows,
                                          float* __restrict__ cnt) {
    const int lane = threadIdx.x & 31;
    const int64_t u = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (u >= n_users) return;
    const int64_t b = u_ptr[u], e = u_ptr[u + 1];
    const float w = isq[u];
    float* row = urows + (size_t)u * 3 * FP;
    for (int c = lane; c < FP; c += 32) {
        float acc = 0.f;
        for (int64_t a = b; a < e; ++a) acc += yj[(size_t)ui_idx[a] * FP + c];
        row[FP + c] = acc * w;
        row[2 * FP + c] = 0.f;
    }
    if (lane == 0) cnt[u] = 0.f;
}

// y_j <- y_j d^{c_j} + lr (1 - d^{c_j}) / (c_j (1 - d)) sum_{u in U_j} g_u,  d = 1 - lr reg,  c_j = sum_{u in U_j} cnt_u: what the reference's
// per-rating updates y_j += lr (err q / sqrt|I_u| - reg y_j) (matrix_factorization.pyx:496-498) add up
// to over the ratings processed since the last application, with the decay applied exactly.
// The c decays and the gradient instalments interleave in the reference; with the instalments spread evenly over
// the c events their decayed sum is acc / c * sum_{k<c} d^k = acc * (1 - d^c) / (c (1 - d)).  For a popular item
// c * lr * reg >> 1 within one epoch, and the undamped sum overshoots several-fold.
__device__ __forceinline__ void svdpp_decay_gain(float c, float lr, float reg, float* decay, float* gain) {
    const float lg = c * log1pf(-lr * reg);
    *decay = expf(lg);
    const float x = c * lr * reg;
    *gain = x > 0.f ? lr * (-expm1f(lg)) / x : lr;  // reg == 0: no decay, plain sum
}

__global__ void svdpp_item_apply_kernel(int64_t n_items, int FP, const int64_t* __restrict__ i_ptr,
                                        const int32_t* __restrict__ iu_idx, const float* __restrict__ urows,
                                        const float* __restrict__ cnt, float lr, float reg, float* __restrict__ yj) {
    const int lane = threadIdx.x & 31;
    const int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (j >= n_items) return;
    const int64_t b = i_ptr[j], e = i_ptr[j + 1];
    float c = 0.f;
    for (int64_t a = b + lane; a < e; a += 32) c += cnt[iu_idx[a]];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    if (c == 0.f) return;
    float decay, gain;
    svdpp_decay_gain(c, lr, reg, &decay, &gain);
    for (int col = lane; col < FP; col += 32) {
        float acc = 0.f;
        for (int64_t a = b; a < e; ++a) acc += urows[(size_t)iu_idx[a] * 3 * FP + 2 * FP + col];
        yj[(size_t)j * FP + col] = yj[(size_t)j * FP + col] * decay + gain * acc;
    }
}

// Ring over P ranks: every rank holds the raters of item j that it owns, so the two sums of the application are
// split -- this kernel writes the rank's partial [sum g_u | sum cnt_u] per item into xch (n_items x (FP + 1)), the
// host all-reduces xch over the ranks (NCCL), svdpp_item_apply_xch_kernel finishes.  y_j is replicated.
__global__ void svdpp_item_partial_kernel(int64_t n_items, int FP, const int64_t* __restrict__ i_ptr,
                                          const int32_t* __restrict__ iu_idx, const float* __restrict__ urows,
                                          const float* __restrict__ cnt, float* __restrict__ xch) {
    const int lane = threadIdx.x & 31;
    const int64_t j = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (j >= n_items) return;
    const int64_t b = i_ptr[j], e = i_ptr[j + 1];
    float c = 0.f;
    for (int64_t a = b + lane; a < e; a += 32) c += cnt[iu_idx[a]];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
    float* out = xch + (size_t)j * (FP + 1);
    for (int col = lane; col < FP; col += 32) {
        float acc = 0.f;
        for (int64_t a = b; a < e; ++a) acc += urows[(size_t)iu_idx[a] * 3 * FP + 2 * FP + col];
        out[col] = acc;
    }
    if (lane == 0) out[FP] = c;
}
__global__ void svdpp_item_apply_xch_kernel(int64_t n_items, int FP, const float* __restrict__ xch, float lr, float reg,
                                            float* __restrict__ yj) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_items * FP) return;
    const int64_t j = t / FP;
    const int col = (int)(t - j * FP);
    const float c = xch[(size_t)j * (FP + 1) + FP];
    if (c == 0.f) return;
    float decay, gain;
    svdpp_decay_gain(c, lr, reg, &decay, &gain);
    yj[t] = yj[t] * decay + gain * xch[(size_t)j * (FP + 1) + col];
}

__global__ void svdpp_isq_kernel(int64_t n_users, const int64_t* __restrict__ u_ptr, float* __restrict__ isq) {
    const int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (u < n_users) {
        const double n = (double)(u_ptr[u + 1] - u_ptr[u]);
        isq[u] = n > 0 ? (float)(1.0 / sqrt(n)) : 0.f;
    }
}
// item -> raters CSR of THIS rank's users: key = item id for the ratings of users u % P == rank, n_items (sorts last)
// for the others; counts per item
__global__ void svdpp_item_key_kernel(int64_t n, const int32_t* __restrict__ u, const int32_t* __restrict__ i, int P,
                                      int rank, int n_items, int* __restrict__ key, int* __restrict__ perm,
                                      unsigned long long* cnt) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    perm[k] = (int)k;
    if (u[k] % P != rank) {
        key[k] = n_items;
        return;
    }
    key[k] = i[k];
    atomicAdd(&cnt[i[k]], 1ull);
}
__global__ void svdpp_gather_users_kernel(int64_t n, const int* __restrict__ perm, const int32_t* __restrict__ u, int P,
                                          int32_t* __restrict__ out) {
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < n) out[k] = u[perm[k]] / P;
}
// ur CSR of the rank's users (local user l = global user rank + l P) cut out of the global ur CSR
__global__ void ring_user_len_kernel(int64_t nu_loc, int P, int rank, const int64_t* __restrict__ u_ptr,
                                     int64_t* __restrict__ len) {
    const int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (l < nu_loc) len[l] = u_ptr[rank + l * P + 1] - u_ptr[rank + l * P];
    if (l == nu_loc) len[l] = 0;
}
__global__ void ring_user_copy_kernel(int64_t nu_loc, int P, int rank, const int64_t* __restrict__ u_ptr,
                                      const int32_t* __restrict__ ui_idx, const int64_t* __restrict__ loc_ptr,
                                      int32_t* __restrict__ loc_idx) {
    const int lane = threadIdx.x & 31;
    const int64_t l = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (l >= nu_loc) return;
    const int64_t src = u_ptr[rank + l * P], dst = loc_ptr[l], len = loc_ptr[l + 1] - dst;
    for (int64_t a = lane; a < len; a += 32) loc_idx[dst + a] = ui_idx[src + a];
}
__global__ void rows_to_f64_kernel(int64_t rows, int f, int stride, const float* __restrict__ src, double* __restrict__ dst) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= rows * f) return;
    const int64_t row = t / f;
    const int c = (int)(t % f);
    dst[t] = (double)src[row * stride + c];
}
__global__ void f32_to_f64_kernel(int64_t n, const float* __restrict__ src, double* __restrict__ dst) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < n) dst[t] = (double)src[t];
}

}  // namespace sb2

// ------------------------------------------------------------------------------------------------
// plan object (C-ABI handle)
// ------------------------------------------------------------------------------------------------
struct sb2_svd_plan {
    int64_t n_users = 0, n_items = 0, n = 0;  // the GLOBAL shape
    // ring over P ranks (P == 1: one GPU): this rank owns users u % P == rank (nu_loc of them) and starts with item
    // super-block `rank`; ni_max = rows of the largest super-block
    int P = 1, rank = 0, device = 0;
    int64_t nu_loc = 0, ni_max = 0, n_loc = 0;
    sb2_sgd_params prm;
    int B = 0, W = 0, G = 0, CH = 0, FP = 0;  // W lane-groups of G lanes, CH 128-bit chunks per lane (0: strided)
    bool stage_u = false, stage_i = false, fast = true;
    bool dep_mode = false;  // dependency-driven cells (one warp per rating, per-row version counters) instead of waves
    size_t smem = 0;
    int *ul = nullptr, *il = nullptr, *off = nullptr, *wave_off = nullptr, *flags = nullptr, *status = nullptr;
    int* dep = nullptr;
    int rec_cap = 0, max_cell = 0;
    int C = 1, ibuf = 0;  // cluster size, floats per item buffer
    float *r = nullptr, *pu = nullptr, *qi = nullptr, *bu = nullptr, *bi = nullptr;
    // SVD++ state
    bool with_yj = false;
    int US = 0, chunks = 1;
    float *yj = nullptr, *isq = nullptr, *cnt = nullptr;
    int64_t *u_ptr = nullptr, *i_ptr = nullptr;
    int32_t *ui_idx = nullptr, *iu_idx = nullptr;
    cudaStream_t alloc_stream = nullptr;
    long long* prof = nullptr;
    // ring state (P > 1): one cudaMalloc'd slab (exportable with cudaIpcGetMemHandle), same layout on every rank:
    // [qi: 2 x ni_max x FP | bi: 2 x ni_max | rflags: B | credit: B]
    void* slab = nullptr;
    size_t slab_bytes = 0;
    void *left_slab = nullptr, *right_slab = nullptr;
    bool left_ipc = false, right_ipc = false;
    int E_done = 0;  // sub-epochs run since the last reset

    int64_t ni_of(int sb) const { return (n_items - sb + P - 1) / P; }
    size_t slab_qi_floats() const { return (size_t)ni_max * FP; }
    float* slab_qi(void* base, int par) const { return reinterpret_cast<float*>(base) + (size_t)par * slab_qi_floats(); }
    float* slab_bi(void* base, int par) const {
        return reinterpret_cast<float*>(base) + 2 * slab_qi_floats() + (size_t)par * ni_max;
    }
    int* slab_rflags(void* base) const { return reinterpret_cast<int*>(slab_bi(base, 0) + 2 * (size_t)ni_max); }
    int* slab_credit(void* base) const { return slab_rflags(base) + B; }
};

namespace sb2 {

typedef void (*dsgd_kernel_t)(const DsgdArgs);

template <int G, int CH>
static dsgd_kernel_t dsgd_kernel_g(const sb2_svd_plan* p) {
    // staging plans: both blocks in shared memory, item block only, or neither.  SVD++ is always biased.
    if (p->with_yj) {
        if (p->stage_u && p->stage_i) return dsgd_svd_kernel<G, CH, true, true, true, true>;
        if (p->stage_i) return dsgd_svd_kernel<G, CH, false, true, true, true>;
        return dsgd_svd_kernel<G, CH, false, false, true, true>;
    }
    const bool b = p->prm.biased != 0;
    if (p->stage_u && p->stage_i)
        return b ? dsgd_svd_kernel<G, CH, true, true, true, false> : dsgd_svd_kernel<G, CH, true, true, false, false>;
    if (p->stage_i)
        return b ? dsgd_svd_kernel<G, CH, false, true, true, false> : dsgd_svd_kernel<G, CH, false, true, false, false>;
    return b ? dsgd_svd_kernel<G, CH, false, false, true, false> : dsgd_svd_kernel<G, CH, false, false, false, false>;
}

// instantiated (G, CH): G is the power of two >= F4 / 4, so CH = ceil(F4 / G) is 3 or 4 (1..4 for G = 1)
static bool dsgd_shape_ok(int g, int ch) {
    if (g == 1) return ch >= 1 && ch <= 4;
    return (g == 2 || g == 4 || g == 8 || g == 16) && (ch == 3 || ch == 4);
}

static dsgd_kernel_t dsgd_kernel(const sb2_svd_plan* p) {
    if (p->dep_mode) {  // G = 32, rows staged, plain SVD
        const bool b = p->prm.biased != 0;
        if (p->CH == 1)
            return b ? dsgd_svd_kernel<32, 1, true, true, true, false, true> : dsgd_svd_kernel<32, 1, true, true, false, false, true>;
        return b ? dsgd_svd_kernel<32, 2, true, true, true, false, true> : dsgd_svd_kernel<32, 2, true, true, false, false, true>;
    }
    if (!p->fast) return dsgd_kernel_g<32, 0>(p);
#define SB2_DSGD_CASE(g, ch) \
    if (p->G == g && p->CH == ch) return dsgd_kernel_g<g, ch>(p);
    SB2_DSGD_CASE(1, 1) SB2_DSGD_CASE(1, 2) SB2_DSGD_CASE(1, 3) SB2_DSGD_CASE(1, 4) SB2_DSGD_CASE(2, 3) SB2_DSGD_CASE(2, 4)
    SB2_DSGD_CASE(4, 3) SB2_DSGD_CASE(4, 4) SB2_DSGD_CASE(8, 3) SB2_DSGD_CASE(8, 4) SB2_DSGD_CASE(16, 3) SB2_DSGD_CASE(16, 4)
#undef SB2_DSGD_CASE
    return nullptr;
}

static void dsgd_launch_config(const sb2_svd_plan* p, int n_blocks, cudaLaunchConfig_t* cfg, cudaLaunchAttribute* attr,
                               cudaStream_t st) {
    memset(cfg, 0, sizeof(*cfg));
    cfg->gridDim = dim3(n_blocks);
    cfg->blockDim = dim3(p->W * p->G);
    cfg->dynamicSmemBytes = p->smem;
    cfg->stream = st;
    int na = 0;
    // Every CTA must be resident: they wait on each other.  Without clusters the cooperative-launch attribute
    // guarantees it.  With clusters the grid is capped at cudaOccupancyMaxActiveClusters instead: the combination
    // cooperative + cluster launch fails under Nsight Compute (LaunchFailed), and a kernel that cannot be
    // profiled is not acceptable here; SB2_DSGD_COOP=1 forces the attribute for cluster launches too.  If the SMs
    // are not free after all (another persistent kernel, an MPS peer), the bounded waits of the kernel (SpinGuard)
    // turn the would-be hang into SB2_ERR_CUDA.
    if (p->C == 1 || getenv("SB2_DSGD_COOP") != nullptr) {
        attr[na].id = cudaLaunchAttributeCooperative;
        attr[na].val.cooperative = 1;
        ++na;
    }
    if (p->C > 1) {
        attr[na].id = cudaLaunchAttributeClusterDimension;
        attr[na].val.clusterDim.x = p->C;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        ++na;
    }
    cfg->attrs = attr;
    cfg->numAttrs = na;
}

static int dsgd_launch(const sb2_svd_plan* p, const DsgdArgs& a, cudaStream_t st) {
    dsgd_kernel_t kern = dsgd_kernel(p);
    SB2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem));
    SB2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, p->C > 8 ? 1 : 0));
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[2];
    dsgd_launch_config(p, p->B, &cfg, attr, st);
    void* args[] = {(void*)&a};
    SB2_CUDA(cudaLaunchKernelExC(&cfg, (const void*)kern, args));
    launch_counter()++;
    return SB2_OK;
}

static void free_async(void* q, cudaStream_t st) {
    if (q) cudaFreeAsync(q, st);
}

// Ring slabs and peer mappings are cached for the life of the process: cudaMalloc / cudaFree of an IPC-exported
// allocation and cudaIpcOpenMemHandle / cudaIpcCloseMemHandle cost milliseconds to hundreds of milliseconds, which
// a fit of 12 ms cannot afford per call.  A destroyed plan returns its slab to the free list; a new plan takes a free
// slab that is large enough (plans alive at the same time -- the ranks of a single-process test ring -- get distinct
// slabs); a peer's handle is opened once and the mapping reused by later fits.
struct RingSlab { void* ptr; size_t bytes; int device; bool in_use; };
static std::mutex g_ring_mu;
static std::vector<RingSlab> g_ring_slabs;
static std::map<std::string, void*> g_ring_peers;   // key: device + 64-byte IPC handle

static cudaError_t ring_slab_acquire(size_t bytes, int device, void** out, size_t* got) {
    std::lock_guard<std::mutex> lk(g_ring_mu);
    for (auto& s : g_ring_slabs)
        if (!s.in_use && s.device == device && s.bytes >= bytes) {
            s.in_use = true; *out = s.ptr; *got = s.bytes;
            return cudaSuccess;
        }
    void* q = nullptr;
    const size_t want = std::max<size_t>(bytes, (size_t)1 << 20);
    cudaError_t e = cudaMalloc(&q, want);
    if (e != cudaSuccess) return e;
    g_ring_slabs.push_back(RingSlab{q, want, device, true});
    *out = q; *got = want;
    return cudaSuccess;
}
static void ring_slab_release(void* q) {
    std::lock_guard<std::mutex> lk(g_ring_mu);
    for (auto& s : g_ring_slabs)
        if (s.ptr == q) s.in_use = false;
}
static cudaError_t ring_peer_open(const unsigned char* h64, int device, void** out) {
    std::lock_guard<std::mutex> lk(g_ring_mu);
    std::string key((const char*)h64, 64);
    key.push_back((char)device);
    auto it = g_ring_peers.find(key);
    if (it != g_ring_peers.end()) { *out = it->second; return cudaSuccess; }
    cudaIpcMemHandle_t h;
    memcpy(&h, h64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess);
    if (e == cudaSuccess) g_ring_peers[key] = *out;
    return e;
}

static void plan_free(sb2_svd_plan* p) {
    if (!p) return;
    cudaStream_t st = p->alloc_stream;
    free_async(p->ul, st); free_async(p->il, st); free_async(p->off, st); free_async(p->wave_off, st); free_async(p->flags, st);
    free_async(p->r, st); free_async(p->prof, st); free_async(p->status, st); free_async(p->dep, st);
    free_async(p->yj, st); free_async(p->isq, st); free_async(p->cnt, st); free_async(p->u_ptr, st);
    free_async(p->i_ptr, st); free_async(p->ui_idx, st); free_async(p->iu_idx, st);
    free_async(p->pu, st); free_async(p->qi, st); free_async(p->bu, st); free_async(p->bi, st);
    if (p->slab) {   // back to the free list (peer mappings stay open: see ring_slab_acquire)
        cudaStreamSynchronize(st);
        ring_slab_release(p->slab);
    }
    delete p;
}

// u, i, r: DEVICE arrays, the all_ratings COO of the WHOLE trainset (every rank of a ring passes the same arrays and
// keeps the ratings of its own users); u_ptr / ui_idx: the global ur CSR (SVD++ only)
int svd_plan_create_dev(int64_t n_users, int64_t n_items, int64_t n, const int32_t* u, const int32_t* i,
                        const double* r, const sb2_sgd_params* prm, int with_yj, const int64_t* u_ptr,
                        const int32_t* ui_idx, int rank, int world, cudaStream_t st, sb2_svd_plan** out) {
    if (with_yj && (!u_ptr || !ui_idx)) {
        set_error("svdpp plan: the ur CSR (u_ptr, ui_idx) is required");
        return SB2_ERR_INVALID;
    }
    if (n_users <= 0 || n_items <= 0 || n < 0 || n > 0x7FFFFFF0ll || prm->n_factors <= 0 || prm->n_factors > 1024) {
        set_error("svd_plan: invalid shape");
        return SB2_ERR_INVALID;
    }
    if (world < 1 || rank < 0 || rank >= world || world > n_users || world > n_items) {
        set_error("svd_plan: invalid rank %d of %d", rank, world);
        return SB2_ERR_INVALID;
    }
    sb2_svd_plan* p = new sb2_svd_plan();
    p->n_users = n_users; p->n_items = n_items; p->n = n; p->prm = *prm;
    p->P = world; p->rank = rank;
    cudaGetDevice(&p->device);
    const int P = world;
    p->nu_loc = (n_users - rank + P - 1) / P;
    p->ni_max = ceil_div(n_items, P);
    const int64_t nu_max = ceil_div(n_users, P);  // sizes that must agree on every rank use the per-rank maxima
    p->alloc_stream = st;
    p->with_yj = with_yj != 0;
    const int f = prm->n_factors;
    p->FP = (int)round_up(f, 4);
    p->US = p->with_yj ? 3 * p->FP : p->FP;
    const int F4 = p->FP / 4;
    // lanes per rating: G = the power of two >= F4 / 4 (at most 16), CH = ceil(F4 / G) <= 4 chunks of 128 bits per
    // lane, rows in registers; rows longer than 256 floats fall back to 32 lanes striding the row.  Fewer, fatter
    // lanes win: with ~13 ratings per wave the critical path is one warp's instruction stream either way, and
    // wider groups only add shuffle steps and warps per scheduler (measured at f = 100: G = 8 / 16 / 32 ->
    // 11.7 / 13.1 / 13.8 ms per fit; f = 20: G = 2 / 4 -> 76 / 87 ms at the ml-10M shape; profiles/r1_summary.md).
    // SB2_DSGD_DEP=1: dependency-driven cells, one warp per rating (DEP kernels; plain SVD, rows of at most 256
    // floats).  An experiment that did not pay (DESIGN.md section 10): a cell then costs its dependency chain or its
    // work / n_warps instead of (waves) x (slowest warp + barrier), but one rating on one warp still takes ~0.9k
    // cycles end to end, and the polling warps compete with the working ones: 14.0 ms per fit (16 warps) against
    // 11.0 ms for the wave kernels at config 2.  Kept selectable, off by default; same results either way.
    p->dep_mode = false;
    if (const char* e = getenv("SB2_DSGD_DEP")) p->dep_mode = atoi(e) != 0 && !p->with_yj && F4 <= 64;
    auto choose_lanes = [&]() {
        p->fast = F4 <= 64;
        p->G = 32;
        p->CH = 0;
        if (p->dep_mode) {
            p->CH = (F4 + 31) / 32;
        } else if (p->fast) {
            int g = 1;
            while (g < 16 && 4 * g < F4) g <<= 1;
            p->G = g;
            p->CH = (F4 + g - 1) / g;
            if (const char* e = getenv("SB2_DSGD_LANES")) {
                const int ge = atoi(e);
                if (ge > 0 && dsgd_shape_ok(ge, (F4 + ge - 1) / ge)) { p->G = ge; p->CH = (F4 + ge - 1) / ge; }
            }
        }
        const int threads = p->dep_mode ? 256 : dsgd_threads(p->G);
        p->W = threads / p->G;
        if (const char* e = getenv("SB2_DSGD_GROUPS")) {
            const int w = atoi(e);
            if (w > 0 && w * p->G <= dsgd_threads(p->G) && (w * p->G) % 32 == 0) p->W = w;
        }
    };
    choose_lanes();
    // Blocks B (= CTAs = strata per sub-epoch) and cluster size C.  With thread-block clusters an item block hops
    // CTA -> CTA through distributed shared memory (~1k cycles) and only every C-th hop goes through L2
    // (~8k cycles), so small cells are affordable: B = K * C as large as the co-residency limit allows, but at
    // least ~16 ratings per cell.  Without clusters (C = 1: rows too long for two smem buffers, or tiny inputs)
    // every hop is an L2 hop and bigger cells win: B ~ sqrt(N / (10 W)).
    // Ring over P ranks: an epoch is P * B strata of (P B)^2 cells, so the chain of strata -- which is what bounds
    // the fit, not the arithmetic -- keeps its single-GPU length when the ranks share the single-GPU block count:
    // B ~ B_1 / P (at least 16).  Every rank derives B and C from the global shape alone, so they agree.
    int B = sm_count();
    int C = 1;
    const int b_rows = (int)std::min<int64_t>(std::min(nu_max, p->ni_max), 1 << 20);
    const size_t budget = 200 * 1024;
    auto plan_smem = [&](int Bc, int Cc, bool* st_i, bool* st_u, size_t* used, int* ibuf) {
        const int mul = (int)ceil_div(nu_max, Bc), mil = (int)ceil_div(p->ni_max, Bc);
        const size_t fixed = (size_t)(2 * (NW + 1) + 2 * P * Bc) * 4 + 64 + (p->dep_mode ? (size_t)(mul + mil) * 4 : 0);
        *ibuf = (int)round_up((int64_t)mil * (p->FP + 1), 4);
        const size_t need_i = (size_t)(Cc > 1 ? 2 : 1) * *ibuf * sizeof(float) + 16;
        const size_t need_u = (size_t)mul * (p->US + 3) * sizeof(float) + 16;
        const size_t min_rec = 256 * 32;
        *st_i = fixed + min_rec + need_i <= budget;
        *st_u = *st_i && fixed + min_rec + need_i + need_u <= budget;
        *used = fixed + (*st_i ? need_i : 0) + (*st_u ? need_u : 0);
    };
    size_t smem_used = 0;
    int b_lim;
    bool b_forced = false;
    {
        const int b_cells = std::max(1, (int)sqrt((double)std::max<int64_t>(n, 1) / 16.0));
        int b_tot = std::min(B, b_cells);
        if (P > 1) b_tot = std::max(b_tot / P, std::min(16, b_tot));
        b_lim = std::min(b_tot, b_rows);
        if (const char* e = getenv("SB2_DSGD_BLOCKS")) {
            const int b = atoi(e);
            if (b > 0 && b <= sm_count()) { b_lim = std::min(b, b_rows); b_forced = true; }
        }
    }
    // largest cluster size (16 is the non-portable maximum, 7 such clusters are co-resident on a B200) that
    // leaves at least two clusters, fits two item buffers in shared memory and passes the occupancy query.
    // Clusters hand item blocks through shared memory only, so the two buffers must fit at the B the plan finally
    // runs with: capping B at the co-resident clusters makes the item blocks larger (27 000 items, f = 100:
    // B 144 -> 112, 188 -> 242 rows), and a cluster size whose buffers no longer fit there is rejected.
    int c_first = 16;
    if (const char* e = getenv("SB2_DSGD_CLUSTER")) c_first = atoi(e);
    auto max_active_clusters = [&](int Bc, int Cc) {
        dsgd_kernel_t kern = dsgd_kernel(p);
        int max_clusters = 0;
        cudaLaunchConfig_t cfg;
        cudaLaunchAttribute attr[2];
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(budget + 16 * 1024));
        cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, Cc > 8 ? 1 : 0);
        dsgd_launch_config(p, Bc, &cfg, attr, st);
        cfg.dynamicSmemBytes = budget;
        if (cudaOccupancyMaxActiveClusters(&max_clusters, (const void*)kern, &cfg) != cudaSuccess) {
            cudaGetLastError();
            max_clusters = 0;
        }
        return max_clusters;
    };
    bool clustered = false;
    for (int Cc = 16; Cc >= 2 && !clustered; Cc >>= 1) {
        if (Cc > c_first || b_lim < 2 * Cc) continue;
        int Bc = b_lim / Cc * Cc;
        p->B = Bc; p->C = Cc;
        plan_smem(Bc, Cc, &p->stage_i, &p->stage_u, &smem_used, &p->ibuf);
        if (!p->stage_i) continue;
        const int max_clusters = max_active_clusters(Bc, Cc);
        if (max_clusters < 2) continue;
        if (Bc / Cc > max_clusters) {
            Bc = max_clusters * Cc;
            p->B = Bc;
            plan_smem(Bc, Cc, &p->stage_i, &p->stage_u, &smem_used, &p->ibuf);
            if (!p->stage_i) continue;
            // the staging variant may have changed with B: its kernel must fit as many clusters
            if (max_active_clusters(Bc, Cc) < Bc / Cc) continue;
        }
        B = Bc;
        C = Cc;
        clustered = true;
    }
    if (!clustered) {
        // no clusters: every hop is an L2 hop (~8k cycles) and bigger cells win: B ~ sqrt(N / (10 W))
        C = 1;
        const int b_work = std::max(4, (int)sqrt((double)std::max<int64_t>(n / ((int64_t)P * P), 1) / (10.0 * p->W)));
        B = std::min(std::min(sm_count(), b_rows), b_work);
        if (b_forced) B = b_lim;
    }
    if (B < 1) B = 1;
    p->B = B;
    p->C = C;
    int max_ul = (int)ceil_div(nu_max, B), max_il = (int)ceil_div(p->ni_max, B);
    plan_smem(B, C, &p->stage_i, &p->stage_u, &smem_used, &p->ibuf);
    const size_t n_cells = (size_t)P * B * B;

    auto fail = [&](int rc) { plan_free(p); return rc; };
    if (P > 1 && !p->stage_i) {
        set_error("svd ring: item blocks of %d rows x %d factors do not fit in shared memory", max_il, f);
        return fail(SB2_ERR_UNSUPPORTED);
    }
    if (C > 1 && !p->stage_i) {   // the DSMEM hop copies the item buffer: a cluster without one has nothing to copy
        set_error("svd_plan: clusters of %d CTAs need two item buffers of %d rows x %d factors in shared memory", C,
                  max_il, f);
        return fail(SB2_ERR_UNSUPPORTED);
    }
#define PLAN_CUDA(expr)                                                                        \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return fail(SB2_ERR_CUDA);                                                         \
        }                                                                                      \
    } while (0)
    const size_t n1 = (size_t)std::max<int64_t>(n, 1);
    PLAN_CUDA(cudaMallocAsync(&p->ul, n1 * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->il, n1 * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->r, n1 * 4, st));
    if (p->dep_mode) PLAN_CUDA(cudaMallocAsync(&p->dep, n1 * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->off, (n_cells + 1) * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->wave_off, n_cells * (NW + 1) * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->flags, (size_t)B * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->status, 16, st));
    PLAN_CUDA(cudaMallocAsync(&p->prof, (size_t)B * 8 * 8, st));
    PLAN_CUDA(cudaMallocAsync(&p->pu, (size_t)p->nu_loc * p->US * 4, st));
    PLAN_CUDA(cudaMallocAsync(&p->bu, (size_t)p->nu_loc * 4, st));
    PLAN_CUDA(cudaMemsetAsync(p->status, 0, 16, st));
    PLAN_CUDA(cudaMemsetAsync(p->flags, 0, (size_t)B * 4, st));
    if (P == 1) {
        PLAN_CUDA(cudaMallocAsync(&p->qi, (size_t)n_items * p->FP * 4, st));
        PLAN_CUDA(cudaMallocAsync(&p->bi, (size_t)n_items * 4, st));
    } else {
        p->slab_bytes = (2 * p->slab_qi_floats() + 2 * (size_t)p->ni_max + 2 * (size_t)B) * 4;
        size_t got = 0;
        PLAN_CUDA(ring_slab_acquire(p->slab_bytes, p->device, &p->slab, &got));
        PLAN_CUDA(cudaMemsetAsync(p->slab, 0, p->slab_bytes, st));
    }

    // stratify: cell key -> stable radix sort -> per-cell colouring + counting sort -> wave tables
    unsigned *key = nullptr, *key2 = nullptr;
    int *val = nullptr, *val2 = nullptr, *cnt = nullptr, *status = nullptr;
    uint8_t* color_tmp = nullptr;
    void* tmp = nullptr;
    auto cleanup = [&]() {
        free_async(key, st); free_async(key2, st); free_async(val, st); free_async(val2, st); free_async(cnt, st);
        free_async(status, st); free_async(tmp, st); free_async(color_tmp, st);
    };
#define PREP_CUDA(expr)                                                                        \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            cleanup();                                                                         \
            return fail(SB2_ERR_CUDA);                                                         \
        }                                                                                      \
    } while (0)
    PREP_CUDA(cudaMallocAsync(&key, n1 * 4, st));
    PREP_CUDA(cudaMallocAsync(&key2, n1 * 4, st));
    PREP_CUDA(cudaMallocAsync(&val, n1 * 4, st));
    PREP_CUDA(cudaMallocAsync(&val2, n1 * 4, st));
    PREP_CUDA(cudaMallocAsync(&color_tmp, n1, st));
    PREP_CUDA(cudaMallocAsync(&cnt, (n_cells + 1) * 4, st));
    PREP_CUDA(cudaMallocAsync(&status, 16, st));
    PREP_CUDA(cudaMemsetAsync(cnt, 0, (n_cells + 1) * 4, st));
    PREP_CUDA(cudaMemsetAsync(status, 0, 16, st));
    int end_bit = 1;
    while (((size_t)1 << end_bit) <= n_cells) ++end_bit;  // keys 0 .. n_cells (n_cells = "not mine / invalid")
    size_t tb1 = 0, tb2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb1, key, key2, val, val2, (int)n, 0, end_bit, st);
    cub::DeviceScan::ExclusiveSum(nullptr, tb2, cnt, p->off, (int)(n_cells + 1), st);
    const size_t tb = std::max(tb1, tb2);
    PREP_CUDA(cudaMallocAsync(&tmp, tb + 16, st));
    const size_t mask_bytes = (size_t)(max_ul + max_il) * 12;  // 64-bit colour masks + int tail counters
    if (mask_bytes > 200 * 1024) {
        set_error("svd_plan: %d + %d rows per block exceed the colouring kernel's shared memory", max_ul, max_il);
        cleanup();
        return fail(SB2_ERR_UNSUPPORTED);
    }
    if (n > 0) {
        const unsigned nb = (unsigned)ceil_div(n, 256);
        dsgd_key_kernel<<<nb, 256, 0, st>>>(n, u, i, B, C, P, rank, (int)n_users, (int)n_items, (unsigned)n_cells, key, val,
                                            cnt, status);
        launch_counter()++;
        size_t t1 = tb;
        PREP_CUDA(cub::DeviceRadixSort::SortPairs(tmp, t1, key, key2, val, val2, (int)n, 0, end_bit, st));
        launch_counter()++;
    }
    size_t t2 = tb;
    PREP_CUDA(cub::DeviceScan::ExclusiveSum(tmp, t2, cnt, p->off, (int)(n_cells + 1), st));
    launch_counter()++;
    {
        PREP_CUDA(cudaFuncSetAttribute(dsgd_color_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mask_bytes));
        const unsigned grid = (unsigned)std::min<size_t>(n_cells, (size_t)sm_count() * 32);
        dsgd_color_kernel<<<grid, 32, mask_bytes, st>>>((int)n_cells, B, P, max_ul, max_il, p->off, val2, u, i, r,
                                                        color_tmp, p->ul, p->il, p->r, p->wave_off, p->dep, status);
        launch_counter()++;
    }
    int status_h[4] = {0, 0, 0, 0};
    int n_loc = 0;
    PREP_CUDA(cudaMemcpyAsync(status_h, status, 16, cudaMemcpyDeviceToHost, st));
    PREP_CUDA(cudaMemcpyAsync(&n_loc, p->off + n_cells, 4, cudaMemcpyDeviceToHost, st));
    PREP_CUDA(cudaStreamSynchronize(st));
    PREP_CUDA(cudaGetLastError());
    cleanup();
    if (status_h[0]) {
        set_error("svd_plan: user / item index out of range");
        return fail(SB2_ERR_INVALID);
    }
    p->n_loc = n_loc;
    if (p->dep_mode && (!p->stage_u || !p->stage_i || status_h[2] >= 0xFFFF)) {
        // rows not resident in shared memory, or a row with >= 65535 ratings in one cell: the wave kernels
        p->dep_mode = false;
        choose_lanes();
    }
    if (p->with_yj) {
        // ur CSR of this rank's users, 1/sqrt|I_u|, item -> (local) raters CSR for the y_j application
        const int64_t nu = p->nu_loc;
        PLAN_CUDA(cudaMallocAsync(&p->yj, (size_t)n_items * p->FP * 4, st));
        PLAN_CUDA(cudaMallocAsync(&p->isq, (size_t)nu * 4, st));
        PLAN_CUDA(cudaMallocAsync(&p->cnt, (size_t)nu * 4, st));
        PLAN_CUDA(cudaMallocAsync(&p->u_ptr, (size_t)(nu + 1) * 8, st));
        PLAN_CUDA(cudaMallocAsync(&p->i_ptr, (size_t)(n_items + 1) * 8, st));
        PLAN_CUDA(cudaMallocAsync(&p->ui_idx, n1 * 4, st));
        PLAN_CUDA(cudaMallocAsync(&p->iu_idx, n1 * 4, st));
        PLAN_CUDA(cudaMemsetAsync(p->cnt, 0, (size_t)nu * 4, st));
        unsigned long long* icnt = nullptr;
        int64_t* ulen = nullptr;
        int *perm_in = nullptr, *perm_out = nullptr, *keys_in = nullptr, *keys_out = nullptr;
        void* tmp2 = nullptr;
        auto cleanup2 = [&]() {
            free_async(icnt, st); free_async(ulen, st); free_async(perm_in, st); free_async(perm_out, st);
            free_async(keys_in, st); free_async(keys_out, st); free_async(tmp2, st);
        };
#define PP_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            cleanup2();                                                                        \
            return fail(SB2_ERR_CUDA);                                                         \
        }                                                                                      \
    } while (0)
        PP_CUDA(cudaMallocAsync(&icnt, (size_t)(n_items + 1) * 8, st));
        PP_CUDA(cudaMallocAsync(&ulen, (size_t)(nu + 1) * 8, st));
        PP_CUDA(cudaMallocAsync(&perm_in, n1 * 4, st));
        PP_CUDA(cudaMallocAsync(&perm_out, n1 * 4, st));
        PP_CUDA(cudaMallocAsync(&keys_in, n1 * 4, st));
        PP_CUDA(cudaMallocAsync(&keys_out, n1 * 4, st));
        PP_CUDA(cudaMemsetAsync(icnt, 0, (size_t)(n_items + 1) * 8, st));
        int item_bits = 1;
        while (((int64_t)1 << item_bits) <= n_items) ++item_bits;
        size_t s1 = 0, s2 = 0, s3 = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, s1, reinterpret_cast<int64_t*>(icnt), p->i_ptr, (int)(n_items + 1), st);
        cub::DeviceRadixSort::SortPairs(nullptr, s2, keys_in, keys_out, perm_in, perm_out, (int)n, 0, item_bits, st);
        cub::DeviceScan::ExclusiveSum(nullptr, s3, ulen, p->u_ptr, (int)(nu + 1), st);
        const size_t sb = std::max(std::max(s1, s2), s3);
        PP_CUDA(cudaMallocAsync(&tmp2, sb + 16, st));
        if (P == 1) {
            PP_CUDA(cudaMemcpyAsync(p->u_ptr, u_ptr, (size_t)(n_users + 1) * 8, cudaMemcpyDeviceToDevice, st));
            PP_CUDA(cudaMemcpyAsync(p->ui_idx, ui_idx, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
        } else {
            ring_user_len_kernel<<<(unsigned)ceil_div(nu + 1, 256), 256, 0, st>>>(nu, P, rank, u_ptr, ulen);
            size_t t5 = sb;
            PP_CUDA(cub::DeviceScan::ExclusiveSum(tmp2, t5, ulen, p->u_ptr, (int)(nu + 1), st));
            ring_user_copy_kernel<<<(unsigned)ceil_div(nu * 32, 256), 256, 0, st>>>(nu, P, rank, u_ptr, ui_idx, p->u_ptr,
                                                                                    p->ui_idx);
            launch_counter() += 3;
        }
        svdpp_isq_kernel<<<(unsigned)ceil_div(nu, 256), 256, 0, st>>>(nu, p->u_ptr, p->isq);
        launch_counter()++;
        if (n > 0) {
            const unsigned nb = (unsigned)ceil_div(n, 256);
            svdpp_item_key_kernel<<<nb, 256, 0, st>>>(n, u, i, P, rank, (int)n_items, keys_in, perm_in, icnt);
            size_t t3 = sb;
            PP_CUDA(cub::DeviceRadixSort::SortPairs(tmp2, t3, keys_in, keys_out, perm_in, perm_out, (int)n, 0, item_bits, st));
            svdpp_gather_users_kernel<<<nb, 256, 0, st>>>(n, perm_out, u, P, p->iu_idx);
            launch_counter() += 3;
        }
        size_t t4 = sb;
        PP_CUDA(cub::DeviceScan::ExclusiveSum(tmp2, t4, reinterpret_cast<int64_t*>(icnt), p->i_ptr, (int)(n_items + 1), st));
        launch_counter()++;
        PP_CUDA(cudaStreamSynchronize(st));
        cleanup2();
        // y_j is applied `chunks` times per epoch.  One application per epoch is the schedule that mirrors the
        // reference: it walks the ratings user by user, so a user's own pushes on the y_j of I_u are all present
        // while that user's ratings are processed (here: z_u advanced in the user row) and, for items with many
        // raters, are decayed away by the other users' updates before the user is seen again (here: the
        // exactly-integrated decay of svdpp_item_apply_kernel + the z_u refresh).  Measured against the
        // sequential oracle at the full ml-10M shape (tests/golden/svdpp_oracle_rmse.json): 1 application
        // 0.8381 vs 0.8380; 2..32 applications 0.847..0.866 (the mid-epoch refresh cuts the own-push
        // accumulation short); DESIGN.md "SVD++".
        p->chunks = 1;
        if (const char* e = getenv("SB2_SVDPP_CHUNKS")) {
            const int c = atoi(e);
            if (c >= 1 && P == 1) p->chunks = std::min(c, B);
        }
    }
    // shared-memory plan: wave table + cell offsets, item buffer(s), user block, then as many of a cell's
    // records as still fit (the rest is read from global memory)
    int rec_cap = std::max(status_h[1], 1);
    const size_t rec_bytes = p->dep_mode ? 32 : 24;  // two buffers of (ul, il, r[, dep])
    rec_cap = (int)std::min<size_t>((size_t)round_up(rec_cap, 4), (budget - smem_used) / rec_bytes / 4 * 4);
    p->rec_cap = rec_cap;
    p->max_cell = status_h[1];
    p->smem = smem_used + (size_t)rec_cap * rec_bytes + 64;
    int smem_optin = 0;
    PLAN_CUDA(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device));
    if (p->smem > (size_t)smem_optin) {
        set_error("svd_plan: %zu bytes of shared memory per CTA exceed the device's %d", p->smem, smem_optin);
        return fail(SB2_ERR_UNSUPPORTED);
    }
    *out = p;
    return SB2_OK;
}

// pu0 / qi0 (/ yj0): DEVICE fp64, the WHOLE (n_users x f), (n_items x f) initial matrices; a rank of a ring keeps
// its users' rows and the rows of item super-block `rank`.  Ring: this also clears the mailboxes the neighbours
// write into, so the caller must synchronise the ranks between reset and run (RingSVD: one all-reduce).
int svd_plan_reset_dev(sb2_svd_plan* p, const double* pu0, const double* qi0, const double* yj0, cudaStream_t st) {
    const int f = p->prm.n_factors;
    const int P = p->P, g = p->rank;
    f64_to_rows_kernel<<<(unsigned)ceil_div(p->nu_loc * p->US, 256), 256, 0, st>>>(p->nu_loc, f, p->US, pu0, p->pu, g, P);
    SB2_LAUNCH_CHECK();
    if (P == 1) {
        f64_to_rows_kernel<<<(unsigned)ceil_div(p->n_items * p->FP, 256), 256, 0, st>>>(p->n_items, f, p->FP, qi0, p->qi, 0, 1);
        SB2_LAUNCH_CHECK();
        SB2_CUDA(cudaMemsetAsync(p->bi, 0, (size_t)p->n_items * 4, st));
    } else {
        SB2_CUDA(cudaMemsetAsync(p->slab, 0, p->slab_bytes, st));
        const int64_t ni = p->ni_of(g);
        f64_to_rows_kernel<<<(unsigned)ceil_div(ni * p->FP, 256), 256, 0, st>>>(ni, f, p->FP, qi0, p->slab_qi(p->slab, 0), g, P);
        SB2_LAUNCH_CHECK();
    }
    if (p->with_yj) {
        if (!yj0) {
            set_error("svd_plan_reset: yj required for SVD++");
            return SB2_ERR_INVALID;
        }
        f64_to_rows_kernel<<<(unsigned)ceil_div(p->n_items * p->FP, 256), 256, 0, st>>>(p->n_items, f, p->FP, yj0, p->yj, 0, 1);
        SB2_LAUNCH_CHECK();
        SB2_CUDA(cudaMemsetAsync(p->cnt, 0, (size_t)p->nu_loc * 4, st));
    }
    SB2_CUDA(cudaMemsetAsync(p->bu, 0, (size_t)p->nu_loc * 4, st));
    SB2_CUDA(cudaMemsetAsync(p->flags, 0, (size_t)p->B * 4, st));
    SB2_CUDA(cudaMemsetAsync(p->status, 0, 16, st));
    p->E_done = 0;
    return SB2_OK;
}

static int fill_args(sb2_svd_plan* p, DsgdArgs& a) {
    memset(&a, 0, sizeof(a));
    a.n_users = (int)p->nu_loc; a.n_items = (int)p->n_items; a.B = p->B; a.W = p->W;
    a.f = p->prm.n_factors; a.FP = p->FP; a.US = p->US;
    a.max_ul = (int)ceil_div(ceil_div(p->n_users, p->P), p->B); a.max_il = (int)ceil_div(p->ni_max, p->B);
    a.dep = p->dep;
    if (const char* e = getenv("SB2_DSGD_DEP_SYNC")) a.dep_sync = atoi(e);
    a.ul = p->ul; a.il = p->il; a.r = p->r; a.cell_off = p->off; a.wave_off = p->wave_off; a.rec_cap = p->rec_cap;
    a.pu = p->pu; a.qi = p->qi; a.bu = p->bu; a.bi = p->bi; a.flags = p->flags; a.status = p->status;
    a.bulk_hop = 1;  // SB2_DSGD_HOP=st: the per-lane st.shared::cluster hop (round 1), for A/B timing
    if (const char* e = getenv("SB2_DSGD_HOP")) a.bulk_hop = strcmp(e, "st") != 0;
    a.isq = p->isq; a.cnt = p->cnt;
    a.C = p->C; a.ibuf = p->ibuf;
    const sb2_sgd_params& q = p->prm;
    a.mu = (q.biased || p->with_yj) ? (float)q.global_mean : 0.f;
    a.lr_bu = (float)q.lr_bu; a.lr_bi = (float)q.lr_bi; a.lr_pu = (float)q.lr_pu; a.lr_qi = (float)q.lr_qi;
    a.reg_bu = (float)q.reg_bu; a.reg_bi = (float)q.reg_bi; a.reg_pu = (float)q.reg_pu; a.reg_qi = (float)q.reg_qi;
    a.lr_yj = (float)q.lr_yj; a.reg_yj = (float)q.reg_yj;
    a.prof = p->prof;
    a.P = p->P; a.rank = p->rank; a.E_base = p->E_done; a.n_items_glob = (int)p->n_items;
    if (p->P > 1) {
        if (!p->left_slab || !p->right_slab) {
            set_error("svd ring: the neighbours are not connected (sb2_svd_ring_connect_*)");
            return SB2_ERR_INVALID;
        }
        for (int par = 0; par < 2; ++par) {
            a.ring_qi[par] = p->slab_qi(p->slab, par); a.ring_bi[par] = p->slab_bi(p->slab, par);
            a.left_qi[par] = p->slab_qi(p->left_slab, par); a.left_bi[par] = p->slab_bi(p->left_slab, par);
        }
        a.rflags = p->slab_rflags(p->slab); a.credit = p->slab_credit(p->slab);
        a.left_rflags = p->slab_rflags(p->left_slab); a.right_credit = p->slab_credit(p->right_slab);
    }
    return SB2_OK;
}

int svd_plan_run(sb2_svd_plan* p, int n_epochs, cudaStream_t st) {
    if (n_epochs <= 0) return SB2_OK;
    if (p->n == 0 && p->P == 1) return SB2_OK;
    DsgdArgs a;
    SB2_TRY(fill_args(p, a));
    if (p->P > 1) {
        // ring: one persistent launch for all epochs; the item blocks travel rank -> rank inside the kernel
        if (p->with_yj) {
            set_error("svd ring: SVD++ runs epoch by epoch (sb2_svd_ring_epoch_dev)");
            return SB2_ERR_INVALID;
        }
        a.n_epochs = n_epochs; a.s_begin = 0; a.s_end = p->P * p->B;
        SB2_TRY(dsgd_launch(p, a, st));
        p->E_done += n_epochs * p->P;
        return SB2_OK;
    }
    if (!p->with_yj) {
        int split = 1;  // SB2_DSGD_SPLIT=n: every epoch as n launches over strata ranges (same updates, same order)
        if (const char* e = getenv("SB2_DSGD_SPLIT")) split = std::max(1, std::min(atoi(e), p->B));
        if (split == 1) {
            a.n_epochs = n_epochs; a.s_begin = 0; a.s_end = p->B;
            SB2_CUDA(cudaMemsetAsync(p->flags, 0, (size_t)p->B * 4, st));
            return dsgd_launch(p, a, st);
        }
        for (int ep = 0; ep < n_epochs; ++ep)
            for (int c = 0; c < split; ++c) {
                a.n_epochs = 1;
                a.s_begin = (int)((int64_t)p->B * c / split);
                a.s_end = (int)((int64_t)p->B * (c + 1) / split);
                SB2_CUDA(cudaMemsetAsync(p->flags, 0, (size_t)p->B * 4, st));
                SB2_TRY(dsgd_launch(p, a, st));
            }
        return SB2_OK;
    }
    // SVD++: per epoch `chunks` x { refresh z_u and clear g_u; strata of the chunk; apply g to y_j }
    const unsigned ub = (unsigned)ceil_div(p->n_users * 32, 256), ib = (unsigned)ceil_div(p->n_items * 32, 256);
    for (int ep = 0; ep < n_epochs; ++ep)
        for (int c = 0; c < p->chunks; ++c) {
            a.n_epochs = 1;
            a.s_begin = (int)((int64_t)p->B * c / p->chunks);
            a.s_end = (int)((int64_t)p->B * (c + 1) / p->chunks);
            if (a.s_begin == a.s_end) continue;
            svdpp_user_refresh_kernel<<<ub, 256, 0, st>>>(p->n_users, p->FP, p->u_ptr, p->ui_idx, p->yj, p->isq, p->pu,
                                                          p->cnt);
            SB2_LAUNCH_CHECK();
            SB2_CUDA(cudaMemsetAsync(p->flags, 0, (size_t)p->B * 4, st));
            SB2_TRY(dsgd_launch(p, a, st));
            svdpp_item_apply_kernel<<<ib, 256, 0, st>>>(p->n_items, p->FP, p->i_ptr, p->iu_idx, p->pu, p->cnt, a.lr_yj,
                                                        a.reg_yj, p->yj);
            SB2_LAUNCH_CHECK();
        }
    return SB2_OK;
}

// ---- all ranks of a ring in one launch on one GPU (sb2_svd_ring_run_local: single-GPU tests of the ring) ------------
typedef void (*dsgd_multi_kernel_t)(const DsgdMulti);
static dsgd_multi_kernel_t dsgd_multi_kernel(const sb2_svd_plan* p) {
#define SB2_MULTI_CASE(g, ch)                                                                                   \
    if (p->G == g && p->CH == ch) {                                                                             \
        if (p->with_yj) return dsgd_svd_multi_kernel<g, ch, true, true>;                                        \
        return p->prm.biased ? dsgd_svd_multi_kernel<g, ch, true, false> : dsgd_svd_multi_kernel<g, ch, false, false>; \
    }
    SB2_MULTI_CASE(1, 1) SB2_MULTI_CASE(1, 2) SB2_MULTI_CASE(1, 3) SB2_MULTI_CASE(1, 4) SB2_MULTI_CASE(2, 3) SB2_MULTI_CASE(2, 4)
    SB2_MULTI_CASE(4, 3) SB2_MULTI_CASE(4, 4) SB2_MULTI_CASE(8, 3) SB2_MULTI_CASE(8, 4)
#undef SB2_MULTI_CASE
    return nullptr;
}

// plans[0 .. n): the ranks 0 .. n-1 of one ring, created in this process on the current device and connected with
// sb2_svd_ring_connect_local.  Runs n_epochs epochs of all of them as ONE kernel launch.
int svd_ring_run_local(sb2_svd_plan** plans, int n, int n_epochs, cudaStream_t st) {
    if (n < 1 || n > DSGD_MAX_VIRTUAL || n_epochs <= 0) {
        set_error("svd_ring_run_local: 1..%d ranks, n_epochs > 0", DSGD_MAX_VIRTUAL);
        return SB2_ERR_INVALID;
    }
    sb2_svd_plan* p0 = plans[0];
    DsgdMulti m;
    memset(&m, 0, sizeof(m));
    size_t smem = 0;
    for (int g = 0; g < n; ++g) {
        sb2_svd_plan* p = plans[g];
        if (!p || p->P != n || p->rank != g || p->B != p0->B || p->C != p0->C || p->G != p0->G || p->CH != p0->CH ||
            p->W != p0->W || p->with_yj != p0->with_yj || !p->stage_u || !p->stage_i || p->dep_mode || !p->fast) {
            set_error("svd_ring_run_local: plans must be the ranks 0..n-1 of one ring with both blocks staged in shared memory");
            return SB2_ERR_INVALID;
        }
        SB2_TRY(fill_args(p, m.r[g]));
        m.r[g].n_epochs = n_epochs; m.r[g].s_begin = 0; m.r[g].s_end = p->P * p->B;
        smem = std::max(smem, p->smem);
    }
    dsgd_multi_kernel_t kern = dsgd_multi_kernel(p0);
    if (!kern) {
        set_error("svd_ring_run_local: no single-launch kernel for %d lanes x %d chunks", p0->G, p0->CH);
        return SB2_ERR_UNSUPPORTED;
    }
    SB2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SB2_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, p0->C > 8 ? 1 : 0));
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr[2];
    dsgd_launch_config(p0, n * p0->B, &cfg, attr, st);
    cfg.dynamicSmemBytes = smem;
    if (p0->C > 1) {   // every CTA of every rank must be resident at once
        int max_clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&max_clusters, (const void*)kern, &cfg) != cudaSuccess) {
            cudaGetLastError();
            max_clusters = 0;
        }
        if (max_clusters * p0->C < n * p0->B) {
            set_error("svd_ring_run_local: %d x %d CTAs are not co-resident on this GPU (%d clusters of %d fit)", n,
                      p0->B, max_clusters, p0->C);
            return SB2_ERR_UNSUPPORTED;
        }
    }
    void* args[] = {(void*)&m};
    SB2_CUDA(cudaLaunchKernelExC(&cfg, (const void*)kern, args));
    launch_counter()++;
    for (int g = 0; g < n; ++g) plans[g]->E_done += n_epochs * n;
    return SB2_OK;
}

// One SVD++ epoch of a ring, in two halves around the caller's all-reduce of xch (n_items x (FP + 1) fp32, DEVICE):
//   phase 0: refresh z_u of the rank's users from the (replicated) y_j, run the epoch's P sub-epochs, write the
//            rank's partial [sum_u g_u | sum_u cnt_u] per item into xch;
//   phase 1: apply the all-reduced xch to y_j (identical on every rank afterwards).
int svd_ring_epoch_dev(sb2_svd_plan* p, int phase, float* xch, cudaStream_t st) {
    if (!p->with_yj || !xch) {
        set_error("svd_ring_epoch: SVD++ plan and exchange buffer required");
        return SB2_ERR_INVALID;
    }
    const float lr = (float)p->prm.lr_yj, reg = (float)p->prm.reg_yj;
    if (phase == 1) {
        svdpp_item_apply_xch_kernel<<<(unsigned)ceil_div(p->n_items * p->FP, 256), 256, 0, st>>>(p->n_items, p->FP, xch, lr,
                                                                                                 reg, p->yj);
        SB2_LAUNCH_CHECK();
        return SB2_OK;
    }
    DsgdArgs a;
    SB2_TRY(fill_args(p, a));
    svdpp_user_refresh_kernel<<<(unsigned)ceil_div(p->nu_loc * 32, 256), 256, 0, st>>>(p->nu_loc, p->FP, p->u_ptr, p->ui_idx,
                                                                                       p->yj, p->isq, p->pu, p->cnt);
    SB2_LAUNCH_CHECK();
    a.n_epochs = 1; a.s_begin = 0; a.s_end = p->P * p->B;
    if (p->P == 1) SB2_CUDA(cudaMemsetAsync(p->flags, 0, (size_t)p->B * 4, st));
    SB2_TRY(dsgd_launch(p, a, st));
    p->E_done += p->P;
    svdpp_item_partial_kernel<<<(unsigned)ceil_div(p->n_items * 32, 256), 256, 0, st>>>(p->n_items, p->FP, p->i_ptr,
                                                                                        p->iu_idx, p->pu, p->cnt, xch);
    SB2_LAUNCH_CHECK();
    return SB2_OK;
}

// phase 0 of svd_ring_epoch_dev for all ranks of a ring in this process, the P sub-epochs as one launch
int svd_ring_epoch_local(sb2_svd_plan** plans, int n, float** xch, cudaStream_t st) {
    for (int g = 0; g < n; ++g) {
        sb2_svd_plan* p = plans[g];
        if (!p || !p->with_yj || !xch || !xch[g]) {
            set_error("svd_ring_epoch_local: SVD++ plans and exchange buffers required");
            return SB2_ERR_INVALID;
        }
        svdpp_user_refresh_kernel<<<(unsigned)ceil_div(p->nu_loc * 32, 256), 256, 0, st>>>(p->nu_loc, p->FP, p->u_ptr,
                                                                                           p->ui_idx, p->yj, p->isq, p->pu, p->cnt);
        SB2_LAUNCH_CHECK();
    }
    SB2_TRY(svd_ring_run_local(plans, n, 1, st));
    for (int g = 0; g < n; ++g) {
        sb2_svd_plan* p = plans[g];
        svdpp_item_partial_kernel<<<(unsigned)ceil_div(p->n_items * 32, 256), 256, 0, st>>>(p->n_items, p->FP, p->i_ptr,
                                                                                            p->iu_idx, p->pu, p->cnt, xch[g]);
        SB2_LAUNCH_CHECK();
    }
    return SB2_OK;
}

// outputs: DEVICE fp64.  Ring: the rank's own rows -- users rank, rank + P, .. and the items of super-block `rank`
// (home again after whole epochs) -- in local order; y_j whole.
int svd_plan_read_dev(sb2_svd_plan* p, double* pu, double* qi, double* bu, double* bi, double* yj, cudaStream_t st) {
    const int f = p->prm.n_factors;
    const int64_t ni = p->P > 1 ? p->ni_of(p->rank) : p->n_items;
    const float* qsrc = p->P > 1 ? p->slab_qi(p->slab, p->E_done & 1) : p->qi;
    const float* bsrc = p->P > 1 ? p->slab_bi(p->slab, p->E_done & 1) : p->bi;
    if (pu) {
        rows_to_f64_kernel<<<(unsigned)ceil_div(p->nu_loc * f, 256), 256, 0, st>>>(p->nu_loc, f, p->US, p->pu, pu);
        SB2_LAUNCH_CHECK();
    }
    if (qi) {
        rows_to_f64_kernel<<<(unsigned)ceil_div(ni * f, 256), 256, 0, st>>>(ni, f, p->FP, qsrc, qi);
        SB2_LAUNCH_CHECK();
    }
    if (yj && p->with_yj) {
        rows_to_f64_kernel<<<(unsigned)ceil_div(p->n_items * f, 256), 256, 0, st>>>(p->n_items, f, p->FP, p->yj, yj);
        SB2_LAUNCH_CHECK();
    }
    if (bu) {
        f32_to_f64_kernel<<<(unsigned)ceil_div(p->nu_loc, 256), 256, 0, st>>>(p->nu_loc, p->bu, bu);
        SB2_LAUNCH_CHECK();
    }
    if (bi) {
        f32_to_f64_kernel<<<(unsigned)ceil_div(ni, 256), 256, 0, st>>>(ni, bsrc, bi);
        SB2_LAUNCH_CHECK();
    }
    return SB2_OK;
}

// synchronises the stream; SB2_ERR_CUDA if a wait of the persistent kernel ran into its deadline
int svd_plan_status(sb2_svd_plan* p, cudaStream_t st) {
    int h[4] = {0, 0, 0, 0};
    SB2_CUDA(cudaMemcpyAsync(h, p->status, 16, cudaMemcpyDeviceToHost, st));
    SB2_CUDA(cudaStreamSynchronize(st));
    if (h[3] != 0) {
        set_error("dsgd kernel (SB2_DSGD_CHECK build): two ratings of one wave share a %s row",
                  (h[3] & 1) ? "user" : "item");
        return SB2_ERR_CUDA;
    }
#ifdef SB2_DSGD_CHECK
    fprintf(stderr, "SB2_DSGD_CHECK: %d rating updates checked, no row shared within a wave\n", h[2]);
#endif
    if (h[0] != 0) {
        set_error("dsgd kernel: a wait for a neighbour CTA / rank timed out (CTAs not co-resident, or a peer rank "
                  "is not running); the factors of this fit are invalid");
        return SB2_ERR_CUDA;
    }
    return SB2_OK;
}

void svd_plan_destroy(sb2_svd_plan* p) { plan_free(p); }

// ---- ring plumbing: export / map the neighbours' slabs ---------------------------------------------------------
int svd_ring_ipc_handle(const sb2_svd_plan* p, unsigned char* out64) {
    if (!p->slab) {
        set_error("svd_ring_ipc_handle: not a ring plan (world == 1)");
        return SB2_ERR_INVALID;
    }
    cudaIpcMemHandle_t h;
    SB2_CUDA(cudaIpcGetMemHandle(&h, p->slab));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(out64, &h, 64);
    return SB2_OK;
}
int svd_ring_connect_ipc(sb2_svd_plan* p, const unsigned char* left64, const unsigned char* right64) {
    if (!p->slab) {
        set_error("svd_ring_connect: not a ring plan (world == 1)");
        return SB2_ERR_INVALID;
    }
    SB2_CUDA(ring_peer_open(left64, p->device, &p->left_slab));
    SB2_CUDA(ring_peer_open(right64, p->device, &p->right_slab));   // two ranks: the same handle, the same mapping
    p->left_ipc = p->right_ipc = true;
    return SB2_OK;
}
// neighbours that live in the same process (one process driving several GPUs, or several ranks of a test sharing
// one GPU on different streams)
int svd_ring_connect_local(sb2_svd_plan* p, sb2_svd_plan* left, sb2_svd_plan* right) {
    if (!p->slab || !left->slab || !right->slab || left->B != p->B || right->B != p->B || left->ni_max != p->ni_max) {
        set_error("svd_ring_connect_local: plans are not ranks of the same ring");
        return SB2_ERR_INVALID;
    }
    for (sb2_svd_plan* q : {left, right})
        if (q->device != p->device) {
            cudaError_t e = cudaDeviceEnablePeerAccess(q->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
                set_error("cudaDeviceEnablePeerAccess(%d): %s", q->device, cudaGetErrorString(e));
                return SB2_ERR_CUDA;
            }
            cudaGetLastError();
        }
    p->left_slab = left->slab;
    p->right_slab = right->slab;
    p->left_ipc = p->right_ipc = false;
    return SB2_OK;
}
void svd_ring_info(const sb2_svd_plan* p, int64_t* nu_loc, int64_t* ni_loc, int64_t* n_loc, int* stride) {
    if (nu_loc) *nu_loc = p->nu_loc;
    if (ni_loc) *ni_loc = p->P > 1 ? p->ni_of(p->rank) : p->n_items;
    if (n_loc) *n_loc = p->n_loc;
    if (stride) *stride = p->FP;
}

// cycles spent by each CTA of the last run in {flag wait, block load, updates, write-back}: host array [B][8] (see DsgdArgs::prof)
int svd_plan_profile(const sb2_svd_plan* p, long long* out_host) {
    SB2_CUDA(cudaMemcpy(out_host, p->prof, (size_t)p->B * 8 * 8, cudaMemcpyDeviceToHost));
    return SB2_OK;
}
// algorithmic bytes per rating update: read + write pu[u], qi[i], bu[u], bi[i] at fp32 + (u, i, r)
int64_t svd_plan_bytes_per_update(const sb2_svd_plan* p) {
    const long long f = p->prm.n_factors;
    // SVD++ (per-user batched y_j): + read/write of z_u and g_u with every rating, + one y_j row read (refresh)
    // and one g_u row read (application) per rating and chunk
    if (p->with_yj) return 2ll * (4 * f + 2) * 4 + 12 + 2ll * p->chunks * f * 4;
    return 2ll * (2 * f + 2) * 4 + 12;
}
void svd_plan_grid(const sb2_svd_plan* p, int* b, int* w) {
    if (b) *b = p->B;
    if (w) *w = p->W;
}
void svd_plan_layout(const sb2_svd_plan* p, int* b, int* c, int* g, int* ch, int* w, int* stage_u, int* stage_i,
                     int* dep_mode, int64_t* smem, int* rec_cap, int* max_cell) {
    if (b) *b = p->B;
    if (c) *c = p->C;
    if (g) *g = p->G;
    if (ch) *ch = p->CH;
    if (w) *w = p->W;
    if (stage_u) *stage_u = p->stage_u ? 1 : 0;
    if (stage_i) *stage_i = p->stage_i ? 1 : 0;
    if (dep_mode) *dep_mode = p->dep_mode ? 1 : 0;
    if (smem) *smem = (int64_t)p->smem;
    if (rec_cap) *rec_cap = p->rec_cap;
    if (max_cell) *max_cell = p->max_cell;
}
void svd_plan_dims(const sb2_svd_plan* p, int64_t* n_users, int64_t* n_items, int* f, int* with_yj) {
    *n_users = p->n_users; *n_items = p->n_items; *f = p->prm.n_factors; *with_yj = p->with_yj ? 1 : 0;
}

}  // namespace sb2
