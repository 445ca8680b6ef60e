// Stable LSD radix sort of (key, position) pairs, one 9-bit digit per pass, and the block scan it is built on.
// The kernels live in wordgrad.cu; the word-table gradient (wordgrad.cu) and row interning (intern.cu) run them.
#pragma once
#include "common.cuh"

namespace lstur {
namespace wg {

constexpr int RB = 9, RADIX = 1 << RB;             // radix-sort digit
constexpr int SORT_THREADS = 256, SORT_ITEMS = 8, SORT_CH = SORT_THREADS * SORT_ITEMS;

static inline long long sort_blocks(long long n) { return (n + SORT_CH - 1) / SORT_CH; }

// inclusive scan of one int per thread over a block of 256 threads (sm: 8 ints of shared memory)
__device__ __forceinline__ int block_inclusive_scan_256(int v, int* sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  if (lane == 31) sm[warp] = v;
  __syncthreads();
  int add = 0;
  for (int w = 0; w < warp; ++w) add += sm[w];
  __syncthreads();
  return v + add;
}

// Sorts the n pairs (*keys, *pos) by bits [0, bits) of the keys, stably, in ceil(bits / 9) passes that ping-pong
// between (*keys, *pos) and (*keys_tmp, *pos_tmp); on return *keys / *pos point at the sorted pairs.  A digit is
// (key >> shift) & 511 of the signed key: for a negative key the top pass sees sign copies, which keeps the digits of
// different keys different, so equal keys end up adjacent whatever their sign.  ghist: RADIX * sort_blocks(n) ints,
// bintot: RADIX ints.
int radix_sort_pairs(int** keys, int** pos, int** keys_tmp, int** pos_tmp, long long n, int bits, int* ghist, int* bintot,
                     cudaStream_t st, const char* name);

// rows (n_rows, len), in place: each row -> its exclusive prefix sum; totals[r] = the row's sum.
int exclusive_scan_rows(int* rows, int n_rows, int len, int* totals, cudaStream_t st, const char* name);

}  // namespace wg
}  // namespace lstur
