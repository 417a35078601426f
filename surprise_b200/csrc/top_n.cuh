// The top-N order, shared by the selection (top_n.cu) and the rank counts (top_n_eval.cu) so that the two cannot
// drift: a candidate's value is the one AlgoBase.test gives it, and candidates rank by that value descending
// (-0.0 == 0.0, NaN after every number), ties by ascending inner item id.
#pragma once
#include "common.cuh"

namespace sb2 {

constexpr int SEL_THREADS = 256;

// default_est where code == 1 (impossible), minus the offset, np.minimum(high, .) then np.maximum(low, .)
__device__ __forceinline__ double top_n_value(double s, int code, double def, double offset, double low,
                                              double high) {
    if (code == 1) s = def;
    s = __dsub_rn(s, offset);
    s = high < s ? high : s;   // np.minimum(high, est): est itself on ties (signed zeros) and NaN
    s = low > s ? low : s;     // np.maximum(low, est)
    return s;
}

// order-preserving integer image of a value: -0.0 as +0.0, NaN below every number
__device__ __forceinline__ unsigned long long top_n_key(double v) {
    if (v != v) return 0ull;   // NaN: after every number
    const unsigned long long b = (unsigned long long)__double_as_longlong(__dadd_rn(v, 0.0));   // -0.0 -> +0.0
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// (key desc, item asc)
__device__ __forceinline__ bool top_n_better(unsigned long long ka, int ia, unsigned long long kb, int ib) {
    return ka > kb || (ka == kb && ia < ib);
}

// sorts key/item[0, c) best-first (bitonic, padded to the next power of two, which the arrays must hold); c is
// block-uniform and the block has SEL_THREADS threads
static __device__ void top_n_sort(unsigned long long* key, int* item, int c) {
    int P = 1;
    while (P < c) P <<= 1;
    for (int j = c + threadIdx.x; j < P; j += SEL_THREADS) { key[j] = 0ull; item[j] = 0x7FFFFFFF; }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int x = threadIdx.x; x < P; x += SEL_THREADS) {
                const int y = x ^ j;
                if (y > x) {
                    const unsigned long long kx = key[x], ky = key[y];
                    const int ix = item[x], iy = item[y];
                    const bool swap = (x & k) == 0 ? top_n_better(ky, iy, kx, ix) : top_n_better(kx, ix, ky, iy);
                    if (swap) { key[x] = ky; key[y] = kx; item[x] = iy; item[y] = ix; }
                }
            }
            __syncthreads();
        }
}

}  // namespace sb2
