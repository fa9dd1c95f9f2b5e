// staging.cuh — byte streams are assembled in shared memory and written to HBM as
// aligned 32-bit words, so variable-length records (1..8 byte nodes, S-byte leaves)
// still leave the SM as full, coalesced sectors.
#pragma once

#include "common.cuh"

namespace stb {

// `total` bytes are staged at smem[shift .. shift+total) with shift = (dst offset & 3);
// `dst_aligned` = dst - shift is 4-byte aligned.  All threads of the CTA call this
// after a __syncthreads() that made the staged bytes visible.
template <int THREADS>
__device__ __forceinline__ void copy_out_staged(char* dst_aligned, const uint8_t* smem, uint32_t shift, uint32_t total) {
  if (total == 0) return;
  const uint32_t end = shift + total;
  const uint32_t first_word = shift ? 1u : 0u;
  const uint32_t last_word = end >> 2;  // words [first_word, last_word) lie fully inside
  for (uint32_t w = first_word + threadIdx.x; w < last_word; w += THREADS)
    reinterpret_cast<uint32_t*>(dst_aligned)[w] = reinterpret_cast<const uint32_t*>(smem)[w];
  if (threadIdx.x == 0) {
    if (shift) {
      const uint32_t stop = end < 4u ? end : 4u;
      for (uint32_t k = shift; k < stop; ++k) dst_aligned[k] = (char)smem[k];
    }
    if (last_word >= first_word) {
      const uint32_t from = (last_word << 2) > shift ? (last_word << 2) : shift;
      for (uint32_t k = from; k < end; ++k) dst_aligned[k] = (char)smem[k];
    }
  }
}

}  // namespace stb
