// u8 x u8 -> s32 masked-contraction GEMM on the 5th-gen tensor cores (tcgen05.mma kind::i8),
// operands staged by TMA (128B-swizzled K-major tiles), accumulators in TMEM.
//
// One launch evaluates up to 2 accumulators  acc_j = A_{a(j)}[rows] * B_{b(j)}[cols]^T  (256 x 256 tiles, 2 x 256
// TMEM columns) that share up to 2 distinct A-side and 2 distinct B-side panels (all panels are row-major [n_pad][k_pad] u8, the
// K dimension = the reference's `y` index).  The epilogue folds each accumulator into an fp64 plane:
//     out_j[row][col] = beta_j * out_j[row][col] + alpha_j * (double)acc_j
// which is exact as long as the running value stays below 2^53 (digit recombination, see sim.cu).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace sb2 {

constexpr int GEMM_BM = 128;      // rows of A per tile  (UMMA M)
constexpr int GEMM_BN = 128;      // rows of B per tile  (UMMA N)
constexpr int GEMM_BK = 128;      // K bytes per stage (one 128B swizzle atom)
constexpr int GEMM_UMMA_K = 32;   // K per tcgen05.mma for 8-bit operands
constexpr int GEMM_MAX_PANELS = 4;
constexpr int GEMM_MAX_ACC = 4;
constexpr int GEMM_TILE_BYTES = GEMM_BM * GEMM_BK;  // 16 KB per operand tile per stage
constexpr int GEMM_THREADS = 192;                   // warp0 TMA, warp1 MMA, warps2-5 epilogue

struct GemmParams {
    CUtensorMap a_maps[GEMM_MAX_PANELS];
    CUtensorMap b_maps[GEMM_MAX_PANELS];
    double* out[GEMM_MAX_ACC];
    double alpha[GEMM_MAX_ACC];
    int beta[GEMM_MAX_ACC];
    int acc_a[GEMM_MAX_ACC];
    int acc_b[GEMM_MAX_ACC];
    int na, nb, nacc, stages;
    int num_k_blocks;
    int n_tiles;
    long long ld;          // leading dimension of the fp64 planes
    long long plane_row0;  // global row held by plane row 0 (row-block shards)
};

// Host side -----------------------------------------------------------------------------------------
struct GemmJob {
    const uint8_t* a;  // A-side panel
    const uint8_t* b;  // B-side panel
    double* out;
    double alpha;
    int beta;
};

// Builds tensor maps, batches jobs (<= 2 accumulators, <= 4 operand tiles per stage per launch) and
// launches the tcgen05 kernel once per batch over `tiles` (int2 {row_blk, col_blk}, device array).
// A-side panels have a_rows rows, B-side panels b_rows.
int gemm_u8_tc_run2(const GemmJob* jobs, int n_jobs, int64_t a_rows, int64_t b_rows, int64_t k_pad,
                    const int2* tiles_dev, int n_tiles, int64_t ld, int64_t plane_row0, cudaStream_t st);

// rows (= columns) of an output tile: 256, computed by a CTA pair
int gemm_tile_rows();

// int32 C = A B^T, test hook (tensor-core path and dp4a cross-check path).
int gemm_u8_selftest(int use_tc, int64_t m, int64_t n, int64_t k, const uint8_t* a, const uint8_t* b, int32_t* c,
                     cudaStream_t st);

}  // namespace sb2
