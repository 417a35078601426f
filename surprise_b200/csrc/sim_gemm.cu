// tcgen05 / TMA / TMEM u8 GEMM for the similarity contractions (see sim_gemm.cuh).
//
// Roles (one CTA per SM, CTA pairs = clusters of 2, persistent over a host-built tile list):
//   warp 0 lane 0 : TMA producer  -- cp.async.bulk.tensor.2d.cta_group::2 tiles of 128 rows x 128 B (SWIZZLE_128B)
//   warp 1 lane 0 : MMA issuer (leader CTA only) -- tcgen05.mma.cta_group::2.kind::i8, M=256 N=256 K=32, D in TMEM
//   warps 2..5    : epilogue      -- tcgen05.ld 32x32b.x32 -> fp64 fold into the output planes
// Pipelines: smem ring (full/empty mbarriers, TMA <-> MMA) and one TMEM hand-off (MMA <-> epilogue).
#include <cuda.h>
#include <cuda_runtime.h>

#include <stdlib.h>

#include <vector>

#include "sim_gemm.cuh"

namespace sb2 {

// ----------------------------------------------------------------------------------------------
// PTX wrappers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format, cute::UMMA::SmemDescriptor):
//   [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major, 1) | [32,46) SBO>>4 = 8 rows * 128 B
//   [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
// K advances inside the 128 B swizzle atom by adding the byte offset to the start address (4 MMAs of K = 32 B).
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format S32 (2) @[4,6), a/b format U8 (0)
// @[7,10)/[10,13), K-major both, N>>3 @[17,23), M>>4 @[24,29).
__host__ __device__ constexpr uint32_t make_idesc_u8(int m, int n) {
    return (2u << 4) | (0u << 7) | (0u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

struct GemmSmemLayout {
    // [stages][na+nb] tiles of 8 KB, then barriers
    static __host__ __device__ size_t tiles_bytes(int stages, int npanels) {
        return (size_t)stages * npanels * GEMM_TILE_BYTES;
    }
};

// ==============================================================================================
// tcgen05 cta_group::2: a CTA pair on one TPC computes a 256 x 256 tile.  Each CTA stages its own
// 128 rows of the A-side tiles and its own 128 rows (half) of the B-side tiles, so an MMA of 256x256x32 reads only
// 4 KB + 4 KB of shared memory per CTA per 128 cycles (64 B/clk instead of 128 B/clk for the 1-CTA 128x128 form,
// which together with the TMA refill saturated the 128 B/clk shared-memory port, DESIGN.md section 10).
// Two accumulators of 256 TMEM columns each per launch.  The leader CTA (cluster rank 0) issues every MMA; both
// CTAs' TMA loads complete on the leader's "full" barrier; tcgen05.commit is multicast to both CTAs' "empty" /
// "tmem full" barriers; both CTAs' epilogue warps arrive on the leader's "tmem empty" barrier.
// ==============================================================================================
constexpr int GEMM2_BM = 256, GEMM2_BN = 256;

__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta_rank));
    return r;
}
__device__ __forceinline__ uint32_t cluster_ctarank2() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync2() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the mbarrier of the pair's leader CTA
__device__ __forceinline__ void tma_load_2d_cg2(const CUtensorMap* map, uint32_t leader_bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tc_commit_cg2_mc(uint64_t* bar, uint16_t cta_mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"(cta_mask)
        : "memory");
}
__device__ __forceinline__ void tc_mma_i8_cg2(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_u8_tc_kernel(const __grid_constant__ GemmParams p, const int2* __restrict__ tiles) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int npanels = p.na + p.nb;
    const int stages = p.stages;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + GemmSmemLayout::tiles_bytes(stages, npanels));
    uint64_t* empty_bar = full_bar + stages;
    uint64_t* tmem_full_bar = empty_bar + stages;
    uint64_t* tmem_empty_bar = tmem_full_bar + 1;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank2();
    const int pair_id = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < stages; ++s) {
            mbar_init(&full_bar[s], 1);   // leader producer's arrive.expect_tx (bytes of BOTH CTAs)
            mbar_init(&empty_bar[s], 1);  // one multicast commit from the leader's MMA thread
        }
        mbar_init(tmem_full_bar, 1);
        mbar_init(tmem_empty_bar, 8);     // 4 epilogue warps x 2 CTAs (only the leader's copy is waited on)
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)),
                     "r"(512u));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync2();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    const int nk = p.num_k_blocks;
    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int t = pair_id; t < p.n_tiles; t += n_pairs) {
                const int2 tile = tiles[t];
                for (int kb = 0; kb < nk; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);  // the MMAs that read this slot (in both CTAs) retired
                    if (rank == 0) mbar_expect_tx(&full_bar[stage], (uint32_t)(2 * npanels * GEMM_TILE_BYTES));
                    const uint32_t lbar = mapa_u32(smem_u32(&full_bar[stage]), 0);
                    uint8_t* sbase = smem + (size_t)stage * npanels * GEMM_TILE_BYTES;
                    for (int a = 0; a < p.na; ++a)
                        tma_load_2d_cg2(&p.a_maps[a], lbar, sbase + a * GEMM_TILE_BYTES, kb * GEMM_BK,
                                        tile.x * GEMM2_BM + (int)rank * 128);
                    for (int b = 0; b < p.nb; ++b)
                        tma_load_2d_cg2(&p.b_maps[b], lbar, sbase + (p.na + b) * GEMM_TILE_BYTES, kb * GEMM_BK,
                                        tile.y * GEMM2_BN + (int)rank * 128);
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc = make_idesc_u8(GEMM2_BM, GEMM2_BN);
            int stage = 0;
            uint32_t phase = 0, tphase = 0;
            for (int t = pair_id; t < p.n_tiles; t += n_pairs) {
                mbar_wait(tmem_empty_bar, tphase ^ 1);  // both CTAs' epilogues have drained the accumulators
                tc_fence_after();
                for (int kb = 0; kb < nk; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint32_t sbase = smem_u32(smem + (size_t)stage * npanels * GEMM_TILE_BYTES);
                    for (int j = 0; j < p.nacc; ++j) {
                        const uint32_t sa = sbase + p.acc_a[j] * GEMM_TILE_BYTES;
                        const uint32_t sb = sbase + (p.na + p.acc_b[j]) * GEMM_TILE_BYTES;
#pragma unroll
                        for (int k = 0; k < GEMM_BK / GEMM_UMMA_K; ++k) {
                            const uint64_t ad = make_desc_sw128(sa + k * GEMM_UMMA_K);
                            const uint64_t bd = make_desc_sw128(sb + k * GEMM_UMMA_K);
                            tc_mma_i8_cg2(tmem_base + j * GEMM2_BN, ad, bd, idesc, (kb > 0 || k > 0) ? 1u : 0u);
                        }
                    }
                    tc_commit_cg2_mc(&empty_bar[stage], (uint16_t)3);
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
                tc_commit_cg2_mc(tmem_full_bar, (uint16_t)3);
                tphase ^= 1;
            }
        }
    } else {
        const int q = warp & 3;
        uint32_t tphase = 0;
        const uint32_t leader_tmem_empty = mapa_u32(smem_u32(tmem_empty_bar), 0);
        for (int t = pair_id; t < p.n_tiles; t += n_pairs) {
            const int2 tile = tiles[t];
            mbar_wait(tmem_full_bar, tphase);
            tc_fence_after();
            const long long row = (long long)tile.x * GEMM2_BM + (long long)rank * 128 + q * 32 + lane - p.plane_row0;
            for (int j = 0; j < p.nacc; ++j) {
                double* orow = p.out[j] + row * p.ld + (long long)tile.y * GEMM2_BN;
                const double alpha = p.alpha[j];
                const int beta = p.beta[j];
#pragma unroll 1
                for (int c0 = 0; c0 < GEMM2_BN; c0 += 32) {
                    uint32_t v[32];
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(j * GEMM2_BN + c0);
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
                          "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
                          "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
                          "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                        : "r"(taddr));
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    double2* o2 = reinterpret_cast<double2*>(orow + c0);
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        double2 w;
                        w.x = alpha * (double)(int)v[2 * e];
                        w.y = alpha * (double)(int)v[2 * e + 1];
                        if (beta) {
                            const double2 old = o2[e];
                            w.x = __dadd_rn(old.x, w.x);
                            w.y = __dadd_rn(old.y, w.y);
                        }
                        o2[e] = w;
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(leader_tmem_empty);
            tphase ^= 1;
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync2();  // the leader's MMAs read the peer's shared memory and barriers: leave together
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
    }
}

// ----------------------------------------------------------------------------------------------
// host: tensor maps + batching + launch
// ----------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

static int make_panel_map(CUtensorMap* map, const uint8_t* panel, int64_t rows, int64_t k_pad) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled entry point not available");
        return SB2_ERR_CUDA;
    }
    cuuint64_t dims[2] = {(cuuint64_t)k_pad, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)k_pad};
    cuuint32_t box[2] = {(cuuint32_t)GEMM_BK, (cuuint32_t)GEMM_BM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(panel), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld k_pad=%lld", (int)r, (long long)rows, (long long)k_pad);
        return SB2_ERR_CUDA;
    }
    return SB2_OK;
}

int gemm_tile_rows() { return GEMM2_BM; }

static int launch_batch(GemmParams& prm, const int2* tiles_dev, cudaStream_t st) {
    const int npanels = prm.na + prm.nb;
    int stages = (int)((200 * 1024) / ((size_t)npanels * GEMM_TILE_BYTES));
    if (stages > 8) stages = 8;
    prm.stages = stages;
    const size_t smem = GemmSmemLayout::tiles_bytes(stages, npanels) + (2 * stages + 2) * sizeof(uint64_t) + 16 + 1024;
    static bool attr_set = false;
    if (!attr_set) {
        SB2_CUDA(cudaFuncSetAttribute(gemm_u8_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        attr_set = true;
    }
    int pairs = sm_count() / 2;
    if (pairs > prm.n_tiles) pairs = prm.n_tiles;
    if (pairs < 1) return SB2_OK;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(GEMM_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SB2_CUDA(cudaLaunchKernelEx(&cfg, gemm_u8_tc_kernel, prm, tiles_dev));
    launch_counter()++;
    return SB2_OK;
}

int gemm_u8_tc_run2(const GemmJob* jobs, int n_jobs, int64_t a_rows, int64_t b_rows, int64_t k_pad,
                    const int2* tiles_dev, int n_tiles, int64_t ld, int64_t plane_row0, cudaStream_t st) {
    const int tile_rows = GEMM2_BM;
    if (k_pad % GEMM_BK || a_rows % tile_rows || b_rows % tile_rows) {
        set_error("gemm: unpadded shape");
        return SB2_ERR_INVALID;
    }
    const int max_acc = 2;    // 2 x 256 TMEM columns
    const int max_tiles = 4;  // 16 KB operand tiles per stage -> 3 stages
    int j = 0;
    while (j < n_jobs) {
        GemmParams prm;
        memset(&prm, 0, sizeof(prm));
        const uint8_t* ap[GEMM_MAX_PANELS];
        const uint8_t* bp[GEMM_MAX_PANELS];
        int na = 0, nb = 0, nacc = 0;
        while (j < n_jobs && nacc < max_acc) {
            int ia = -1, ib = -1;
            for (int t = 0; t < na; ++t)
                if (ap[t] == jobs[j].a) ia = t;
            for (int t = 0; t < nb; ++t)
                if (bp[t] == jobs[j].b) ib = t;
            if ((ia < 0 && na == GEMM_MAX_PANELS) || (ib < 0 && nb == GEMM_MAX_PANELS)) break;
            // keep a stage at <= 6 tiles (48 KB) so the ring stays >= 4 deep
            const int add = (ia < 0) + (ib < 0);
            if (nacc > 0 && na + nb + add > max_tiles) break;  // >= 3 (pairs) / 2 (1-CTA) stages of 16 KB tiles
            if (ia < 0) { ia = na; ap[na++] = jobs[j].a; }
            if (ib < 0) { ib = nb; bp[nb++] = jobs[j].b; }
            prm.acc_a[nacc] = ia;
            prm.acc_b[nacc] = ib;
            prm.out[nacc] = jobs[j].out;
            prm.alpha[nacc] = jobs[j].alpha;
            prm.beta[nacc] = jobs[j].beta;
            ++nacc;
            ++j;
        }
        for (int t = 0; t < na; ++t) SB2_TRY(make_panel_map(&prm.a_maps[t], ap[t], a_rows, k_pad));
        for (int t = 0; t < nb; ++t) SB2_TRY(make_panel_map(&prm.b_maps[t], bp[t], b_rows, k_pad));
        prm.na = na;
        prm.nb = nb;
        prm.nacc = nacc;
        prm.num_k_blocks = (int)(k_pad / GEMM_BK);
        prm.n_tiles = n_tiles;
        prm.ld = ld;
        prm.plane_row0 = plane_row0;
        SB2_TRY(launch_batch(prm, tiles_dev, st));
    }
    return SB2_OK;
}

// ----------------------------------------------------------------------------------------------
// test hooks
// ----------------------------------------------------------------------------------------------
__global__ void gemm_u8_dp4a_kernel(const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, int32_t* __restrict__ c,
                                    int64_t m, int64_t n, int64_t k) {
    const int64_t col = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t row = blockIdx.y;
    if (col >= n || row >= m) return;
    const uint32_t* ar = reinterpret_cast<const uint32_t*>(a + row * k);
    const uint32_t* br = reinterpret_cast<const uint32_t*>(b + col * k);
    unsigned acc = 0;
    for (int64_t t = 0; t < k / 4; ++t) acc = __dp4a(ar[t], br[t], acc);
    c[row * n + col] = (int32_t)acc;
}

__global__ void plane_to_i32_kernel(const double* __restrict__ p, int32_t* __restrict__ c, int64_t n) {
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t < n) c[t] = (int32_t)p[t];
}

int gemm_u8_selftest(int use_tc, int64_t m, int64_t n, int64_t k, const uint8_t* a, const uint8_t* b, int32_t* c,
                     cudaStream_t st) {
    const int tr = GEMM2_BM;
    if (m % tr || n % tr || k % GEMM_BK) {
        set_error("selftest: m, n multiples of %d and k multiple of %d required", tr, GEMM_BK);
        return SB2_ERR_INVALID;
    }
    if (!use_tc) {
        dim3 grid((unsigned)ceil_div(n, 128), (unsigned)m);
        gemm_u8_dp4a_kernel<<<grid, 128, 0, st>>>(a, b, c, m, n, k);
        SB2_LAUNCH_CHECK();
        return SB2_OK;
    }
    std::vector<int2> tiles;
    for (int r = 0; r < m / tr; ++r)
        for (int cc = 0; cc < n / tr; ++cc) tiles.push_back(make_int2(r, cc));
    DevBuf tiles_d, plane;
    SB2_TRY(tiles_d.alloc(tiles.size() * sizeof(int2), st));
    SB2_CUDA(cudaMemcpyAsync(tiles_d.p, tiles.data(), tiles.size() * sizeof(int2), cudaMemcpyHostToDevice, st));
    SB2_TRY(plane.alloc((size_t)m * n * sizeof(double), st));
    GemmJob job{a, b, plane.as<double>(), 1.0, 0};
    SB2_TRY(gemm_u8_tc_run2(&job, 1, m, n, k, tiles_d.as<int2>(), (int)tiles.size(), n, 0, st));
    plane_to_i32_kernel<<<(unsigned)ceil_div(m * n, 256), 256, 0, st>>>(plane.as<double>(), c, m * n);
    SB2_LAUNCH_CHECK();
    SB2_CUDA(cudaStreamSynchronize(st));  // tiles vector must outlive the async copy
    return SB2_OK;
}

}  // namespace sb2
