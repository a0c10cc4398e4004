// sd_ranksort.cuh -- the per-row rank machinery shared by the rank tests (sd_ranksum.cu: K6,
// sd_kruskal.cu: K7): order-preserving keys, a warp-aggregated gather of a row's defined cells into
// shared memory, the bitonic sort of those keys and the tie-run searches on the sorted keys.
//
// Keys: the IEEE bit pattern made order-preserving (sign set: all bits flipped; clear: sign bit set),
// after -0.0 is canonicalised to +0.0 (rankdata ties them).  float32 cells are widened to double first
// (exact and order-preserving), so both input types share one key.  +-inf are ordinary keys; kPad
// pads the sort above every key a non-NaN value can have.
#pragma once

#include "sd_common.cuh"

namespace sd {
namespace ranksort {

constexpr uint64_t kPad = ~0ull;

__device__ __forceinline__ uint64_t order_key(double v)
{
    uint64_t u = (uint64_t)__double_as_longlong(v);
    if ((u << 1) == 0) u = 0;                                   // -0.0 -> +0.0
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// first position in keys[0, m) whose key is >= key (strict = false) or > key (strict = true)
__device__ __forceinline__ int search(const uint64_t *keys, int lo, int m, uint64_t key, bool strict)
{
    int len = m - lo;
    while (len > 0) {
        const int half = len >> 1;
        const uint64_t k = keys[lo + half];
        if (k < key || (strict && k == key)) {
            lo += half + 1;
            len -= half + 1;
        } else {
            len = half;
        }
    }
    return lo;
}

// The warp-aggregated gather: every lane with `valid` set stores `key` at its own slot of
// keys[*count, ...), in any order, with one shared atomic per warp.  All 32 lanes of the warp run it
// together (a uniform trip count over the cells); the caller zeroes *count and synchronises before
// the first pass and after the last.  A macro rather than an inline function: as a function it lets
// the compiler reorder two predicate moves in K6's loop, whose SASS is kept as it was.
#define SD_RANKSORT_APPEND(keys, count, lane, valid, key)                          \
    do {                                                                           \
        const unsigned _mask = __ballot_sync(0xffffffffu, (valid));                \
        int _slot = 0;                                                             \
        if ((lane) == 0 && _mask) _slot = atomicAdd((count), __popc(_mask));       \
        _slot = __shfl_sync(0xffffffffu, _slot, 0);                                \
        if (valid) (keys)[_slot + __popc(_mask & ((1u << (lane)) - 1u))] = (key);  \
    } while (0)

// Pads keys[m, npad) with kPad, npad the next power of two >= m, and sorts keys[0, npad) ascending
// with a bitonic network.  Every thread of the CTA calls it; it ends on a barrier.
__device__ __forceinline__ void sort(uint64_t *keys, int m)
{
    int npad = 1;
    while (npad < m) npad <<= 1;
    for (int i = m + threadIdx.x; i < npad; i += blockDim.x) keys[i] = kPad;
    __syncthreads();
    for (int k = 2; k <= npad; k <<= 1) {
        for (int h = k >> 1; h > 0; h >>= 1) {
            for (int t = threadIdx.x; t < (npad >> 1); t += blockDim.x) {
                const int lo = 2 * t - (t & (h - 1)), hi = lo + h;
                const uint64_t a = keys[lo], b = keys[hi];
                if ((a > b) == ((lo & k) == 0)) {
                    keys[lo] = b;
                    keys[hi] = a;
                }
            }
            __syncthreads();
        }
    }
}

}  // namespace ranksort
}  // namespace sd
