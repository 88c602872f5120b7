// Device code shared by the two BWT builders: bwt_build.cu (u32 positions and ranks, n < 2^32) and bwt_build_wide.cu
// (u64, the suffix array sorted in parts).
#pragma once
#include <cstdint>

namespace rbg {

constexpr int kBwtBlock = 256;
constexpr int kBwtK = 27;                          // 27 base-5 digits fit 63 bits

__device__ __forceinline__ uint64_t bwt_code(uint8_t c) { return c == 'A' ? 1 : c == 'C' ? 2 : c == 'G' ? 3 : c == 'T' ? 4 : 0; }

__device__ __forceinline__ uint64_t bwt_item() { return (uint64_t) blockIdx.x * kBwtBlock + threadIdx.x; }

// Item k starts a group of equal keys.
__device__ __forceinline__ bool bwt_is_head(const uint64_t* __restrict__ keys, uint64_t k) { return k == 0 || keys[k] != keys[k - 1]; }

// BWT[i] = T[SA[i] - 1], the terminator's byte at the row of SA = 0.  Pos: the position type of the suffix array.
template <class Pos>
__global__ void __launch_bounds__(kBwtBlock) bwt_gather_kernel(const uint8_t* __restrict__ text, const Pos* __restrict__ sa, uint64_t n,
                                                               uint8_t* __restrict__ bwt) {
    const uint64_t i = bwt_item();
    if (i >= n) return;
    const Pos p = sa[i];
    bwt[i] = text[p ? p - 1 : n - 1];
}

// SA at the first and last row of each of r runs starting at rows starts[0..r); the last run ends at row `end` - 1.
template <class Pos, class Row>
__global__ void __launch_bounds__(kBwtBlock) bwt_samples_kernel(const Row* __restrict__ starts, uint64_t r, uint64_t end,
                                                                const Pos* __restrict__ sa, Pos* __restrict__ sa_first,
                                                                Pos* __restrict__ sa_last) {
    const uint64_t j = bwt_item();
    if (j >= r) return;
    sa_first[j] = sa[starts[j]];
    sa_last[j] = sa[(j + 1 < r ? (uint64_t) starts[j + 1] : end) - 1];
}

}  // namespace rbg
