// scan.cuh — prefix sums and sum reductions over a warp, a CTA, and an array scanned by one CTA.
// The bucket offsets, tile bases, radix-sort rows, serialized byte offsets and rank indexes of the
// library all go through these.
#pragma once

#include "common.cuh"

namespace stb {

// Inclusive prefix sum over the 32 lanes of a full warp.
template <typename T>
__device__ __forceinline__ T warp_inclusive_sum(T v) {
  const uint32_t lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const T y = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += y;
  }
  return v;
}

// Sum over the 32 lanes of a full warp; every lane gets it.
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

// Exclusive prefix sum of v over the THREADS threads of the CTA, all of which call it; the CTA's
// total goes to every thread's *total when total is not null.  warp_totals: THREADS / 32 words of
// shared memory.
// Barriers: exactly one __syncthreads(), between storing the warp totals and reading them, so
// shared-memory stores a caller makes before the call are visible to every thread after it.
// None on entry or exit: warp_totals may be written again (by another call) only after the
// caller's next __syncthreads().
template <int THREADS, typename T>
__device__ __forceinline__ T block_exclusive_sum(T v, T* warp_totals, T* total = nullptr) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const T x = warp_inclusive_sum(v);
  if (lane == 31) warp_totals[warp] = x;
  __syncthreads();
  T before = 0;
  for (uint32_t w = 0; w < warp; ++w) before += warp_totals[w];
  if (total) {
    T sum = before;
    for (uint32_t w = warp; w < THREADS / 32; ++w) sum += warp_totals[w];
    *total = sum;
  }
  return before + x - v;
}

// Exclusive prefix sum of in[0, n) into out[0, n) (in == out scans in place) by one CTA of 1024
// threads, 1024 elements at a time with a carry; returns the total to every thread.  Each element
// is read and written by the same thread.
template <typename T>
__device__ __forceinline__ T cta_exclusive_scan(const T* in, T* out, uint32_t n) {
  __shared__ T warp_totals[32];
  T carry = 0;
  for (uint32_t base = 0; base < n; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    T block_total;
    const T before = block_exclusive_sum<1024>(i < n ? in[i] : T(0), warp_totals, &block_total);
    if (i < n) out[i] = carry + before;
    carry += block_total;
    __syncthreads();  // the next block writes warp_totals again
  }
  return carry;
}

// One CTA of 1024 threads per row: rows[r * n, r * n + n) is scanned in place (exclusive) and its
// total goes to row_totals[r].
template <typename T>
static __global__ void __launch_bounds__(1024) exclusive_scan_rows_kernel(T* rows, uint32_t n, T* row_totals) {
  T* row = rows + (size_t)blockIdx.x * n;
  const T total = cta_exclusive_scan(row, row, n);
  if (threadIdx.x == 0) row_totals[blockIdx.x] = total;
}

}  // namespace stb
