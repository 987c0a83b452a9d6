// block_scan.cuh -- warp and block prefix sums shared by the stream compactions (crop, uniform sampling, GetMap, map export)
// and the warp-level selections of the K-NN builder and the median.
//
// The block-wide helpers assume blocks of SCAN_BLOCK threads (32 full warps).  The library is built without -rdc, one
// object per .cu, so the kernel below has internal linkage: every object that launches it keeps its own instance.
#pragma once
#include <cuda_runtime.h>

namespace svn {

constexpr int SCAN_BLOCK = 1024;

// inclusive prefix sum over the 32 lanes of a full warp
template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T v) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v += u;
  }
  return v;
}

// exclusive prefix sum over the block; the block's total to *total when total is not null.  int, or long long for point offsets
template <typename T>
__device__ T block_exclusive_scan(T v, T *total) {
  __shared__ T s_w[32];
  __shared__ T s_tot;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const T incl = warp_inclusive_scan(v);
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const T x = s_w[lane], xi = warp_inclusive_scan(x);
    s_w[lane] = xi - x;
    if (lane == 31) s_tot = xi;
  }
  __syncthreads();
  const T r = s_w[warp] + incl - v;
  if (total) *total = s_tot;
  __syncthreads();
  return r;
}

// sum of v over the block, stored to *out by thread 0
__device__ __forceinline__ void block_sum_int(int v, int *out) {
  __shared__ int s_w[32];
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    int w = s_w[threadIdx.x];
    for (int o = 16; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
    if (threadIdx.x == 0) *out = w;
  }
}

namespace {

// The middle step of a block-wise compaction (count per block -> this -> emit): one block turns the n_blocks per-block sums
// into their exclusive prefix in place, SCAN_BLOCK at a time with a running carry, and stores the grand total to *total_out.
template <typename T>
__global__ void __launch_bounds__(SCAN_BLOCK) k_scan_block_sums(T *block_sums, int n_blocks, long long *total_out) {
  T carry = 0;
  for (int base = 0; base < n_blocks; base += SCAN_BLOCK) {
    const int i = base + threadIdx.x;
    const T v = i < n_blocks ? block_sums[i] : 0;
    T tot;
    const T ex = block_exclusive_scan(v, &tot);
    if (i < n_blocks) block_sums[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) *total_out = carry;
}

}  // namespace
}  // namespace svn
