// sort.cu — frequency sort of every layer (shared_tree::sort_tree).
//
// Replaces histogram / sort_leaves / sort_nodes / invert_indices / reorder_layer /
// rewire_nodes (reference src/shared_tree.cpp:316-326, :350-483).  The reference sorts
// layer by layer in two std::async waves because each sort_nodes call rewrites two
// layers in place.  Here the dependency is removed instead: every child layer's
// histogram depends only on its parent's *contents* (not its order), so all new
// positions are computed first from the untouched tree, and each layer is then
// permuted and rewired exactly once, out of place:
//
//     new_nodes[k][ newpos[k+1][i] ] = rewire(nodes[k][i], newpos[k])
//
// new position = rank under (frequency desc, old index asc) = a stable LSD radix sort
// of (maxf - freq) over only the digits maxf needs; the last pass scatters the rank
// straight into newpos[].
#include <algorithm>

#include "scan.cuh"
#include "tree.h"

namespace stb {

constexpr int HS_THREADS = 256;

// freq[child index] += 1 for every non-null pointer of the parent layer.
__global__ void __launch_bounds__(HS_THREADS)
histogram_kernel(const uint2* __restrict__ nodes, uint32_t n, uint32_t* __restrict__ freq) {
  const uint32_t i = blockIdx.x * HS_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint2 nd = __ldg(nodes + i);
  if (!ptr_is_null(nd.x)) atomicAdd(freq + (nd.x & IDX_MASK), 1u);
  if (!ptr_is_null(nd.y)) atomicAdd(freq + (nd.y & IDX_MASK), 1u);
}

__global__ void __launch_bounds__(HS_THREADS)
max_kernel(const uint32_t* __restrict__ freq, uint32_t n, uint32_t* __restrict__ out_max, uint32_t* __restrict__ out_min) {
  // both ends of the frequency range: an imported tree may hold unreferenced items (frequency 0).
  // 16-byte loads (the arrays are carved at 256-byte offsets), the tail word by word.
  uint32_t m = 0, lo = 0xffffffffu;
  const uint32_t n4 = n / 4;
  const uint4* v4 = reinterpret_cast<const uint4*>(freq);
  for (uint32_t i = blockIdx.x * HS_THREADS + threadIdx.x; i < n4; i += gridDim.x * HS_THREADS) {
    const uint4 f = __ldg(v4 + i);
    m = max(max(m, f.x), max(f.y, max(f.z, f.w)));
    lo = min(min(lo, f.x), min(f.y, min(f.z, f.w)));
  }
  if (blockIdx.x == 0 && threadIdx.x < n - 4 * n4) {
    const uint32_t f = freq[4 * n4 + threadIdx.x];
    m = max(m, f);
    lo = min(lo, f);
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, d));
  }
  if ((threadIdx.x & 31) == 0) {
    if (m) atomicMax(out_max, m);
    atomicMin(out_min, lo);
  }
}

// ---- stable LSD radix sort, 8-bit digits -----------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_GROUPS = 16;                           // 32-item groups per warp
constexpr int RS_TILE = RS_THREADS * RS_GROUPS;         // 4096 items per CTA
constexpr int RS_WARP_ITEMS = 32 * RS_GROUPS;           // a warp owns 512 consecutive items

__device__ __forceinline__ uint32_t rs_digit(uint32_t freq, uint32_t maxf, int shift) {
  return ((maxf - freq) >> shift) & 0xffu;
}

// Per-CTA digit histogram, written digit-major: hist[d * nblocks + b].
__global__ void __launch_bounds__(RS_THREADS)
radix_hist_kernel(const uint32_t* __restrict__ keys, uint32_t n, uint32_t maxf, int shift, uint32_t nblocks,
                  uint32_t* __restrict__ hist) {
  __shared__ uint32_t bins[256];
  bins[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t warp_base = blockIdx.x * RS_TILE + warp * RS_WARP_ITEMS;
#pragma unroll 4
  for (int g = 0; g < RS_GROUPS; ++g) {
    const uint32_t i = warp_base + g * 32 + lane;
    const bool ok = i < n;
    const uint32_t d = ok ? rs_digit(keys[i], maxf, shift) : 0x100u;
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    if (ok && lane == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&bins[d], (uint32_t)__popc(peers));
  }
  __syncthreads();
  hist[threadIdx.x * nblocks + blockIdx.x] = bins[threadIdx.x];
}

// Scatter pass.  FIRST: values are the implicit identity.  LAST: instead of moving the
// pair, publish the destination rank: newpos[value] = rank.
template <bool FIRST, bool LAST>
__global__ void __launch_bounds__(RS_THREADS)
radix_scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in, uint32_t n,
                     uint32_t maxf, int shift, uint32_t nblocks, const uint32_t* __restrict__ hist,
                     const uint32_t* __restrict__ row_total, uint32_t* __restrict__ keys_out,
                     uint32_t* __restrict__ vals_out) {
  __shared__ uint32_t digit_base[256];            // global offset of (digit, this CTA)
  __shared__ uint32_t warp_cnt[RS_WARPS][256];    // per-warp counts, then running offsets
  __shared__ uint32_t scan_tmp[RS_WARPS];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // exclusive scan of the 256 row totals
  digit_base[threadIdx.x] = block_exclusive_sum<RS_THREADS>(row_total[threadIdx.x], scan_tmp) + hist[threadIdx.x * nblocks + blockIdx.x];
#pragma unroll
  for (int w = 0; w < RS_WARPS; ++w) warp_cnt[w][threadIdx.x] = 0;
  __syncthreads();

  const uint32_t warp_first = blockIdx.x * RS_TILE + warp * RS_WARP_ITEMS;
  uint32_t key[RS_GROUPS];
  // pass 1: per-warp digit counts
#pragma unroll
  for (int g = 0; g < RS_GROUPS; ++g) {
    const uint32_t i = warp_first + g * 32 + lane;
    const bool ok = i < n;
    key[g] = ok ? keys_in[i] : 0u;
    const uint32_t d = ok ? rs_digit(key[g], maxf, shift) : 0x100u;
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    if (ok && lane == (uint32_t)(__ffs(peers) - 1)) warp_cnt[warp][d] += __popc(peers);
    __syncwarp();
  }
  __syncthreads();
  // per digit: exclusive scan over the warps, offset by the CTA's global base
  {
    uint32_t run = digit_base[threadIdx.x];
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
      const uint32_t c = warp_cnt[w][threadIdx.x];
      warp_cnt[w][threadIdx.x] = run;
      run += c;
    }
  }
  __syncthreads();
  // pass 2: stable scatter
#pragma unroll
  for (int g = 0; g < RS_GROUPS; ++g) {
    const uint32_t i = warp_first + g * 32 + lane;
    const bool ok = i < n;
    const uint32_t d = ok ? rs_digit(key[g], maxf, shift) : 0x100u;
    const uint32_t peers = __match_any_sync(0xffffffffu, d);
    uint32_t dst = 0;
    if (ok) dst = warp_cnt[warp][d] + __popc(peers & ((1u << lane) - 1u));
    __syncwarp();
    if (ok && lane == (uint32_t)(__ffs(peers) - 1)) warp_cnt[warp][d] += __popc(peers);
    __syncwarp();
    if (ok) {
      const uint32_t v = FIRST ? i : vals_in[i];
      if (LAST) {
        vals_out[v] = dst;  // newpos[old index] = rank
      } else {
        keys_out[dst] = key[g];
        vals_out[dst] = v;
      }
    }
  }
}

// new_nodes[dst_map ? dst_map[i] : i] = nodes[i] with child indices mapped through
// child_map (identity when null).  Flags are kept; null stays null (shared_tree.cpp:383-403).
__global__ void __launch_bounds__(HS_THREADS)
permute_rewire_kernel(const uint2* __restrict__ nodes, uint32_t n, const uint32_t* __restrict__ child_map,
                      const uint32_t* __restrict__ dst_map, uint2* __restrict__ out) {
  const uint32_t i = blockIdx.x * HS_THREADS + threadIdx.x;
  if (i >= n) return;
  uint2 nd = __ldg(nodes + i);
  if (child_map) {
    if (!ptr_is_null(nd.x)) nd.x = (nd.x & ~IDX_MASK) | __ldg(child_map + (nd.x & IDX_MASK));
    if (!ptr_is_null(nd.y)) nd.y = (nd.y & ~IDX_MASK) | __ldg(child_map + (nd.y & IDX_MASK));
  }
  out[dst_map ? __ldg(dst_map + i) : i] = nd;
}

__global__ void __launch_bounds__(HS_THREADS)
permute_leaves_kernel(const unsigned long long* __restrict__ leaves, uint32_t n, const uint32_t* __restrict__ dst_map,
                      unsigned long long* __restrict__ out) {
  const uint32_t i = blockIdx.x * HS_THREADS + threadIdx.x;
  if (i >= n) return;
  out[__ldg(dst_map + i)] = __ldg(leaves + i);
}

__global__ void widen_kernel(const uint32_t* __restrict__ in, uint32_t n, unsigned long long* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i];
}

// ---- host --------------------------------------------------------------------------

static uint64_t child_count(const Tree& t, uint64_t layer) { return layer == 0 ? t.n_leaves : t.layers[layer - 1].count; }

// freq: child_count(t, layer) words, caller-owned
static int histogram_into(const Tree& t, uint64_t layer, uint32_t* freq) {
  Tree& ctx = const_cast<Tree&>(t);
  const uint64_t n_child = child_count(t, layer);
  STB_CUDA(ctx, cudaMemsetAsync(freq, 0, std::max<uint64_t>(n_child, 1) * 4, t.stream));
  const uint32_t n = (uint32_t)t.layers[layer].count;
  Launch l(ctx, "histogram");
  histogram_kernel<<<(unsigned)ceil_div(n, HS_THREADS), HS_THREADS, 0, t.stream>>>(t.layers[layer].nodes.ptr, n, freq);
  return STB_OK;
}

int histogram_layer(const Tree& t, uint64_t layer, DevBuf<uint32_t>& freq) {
  Tree& ctx = const_cast<Tree&>(t);
  STB_CUDA(ctx, freq.alloc(std::max<uint64_t>(child_count(t, layer), 1), t.stream));
  return histogram_into(t, layer, freq.ptr);
}

int histogram_u64(const Tree& t, uint64_t layer, unsigned long long* d_out) {
  Tree& ctx = const_cast<Tree&>(t);
  DevBuf<uint32_t> freq;
  STB_TRY(histogram_layer(t, layer, freq));
  const uint32_t n = (uint32_t)child_count(t, layer);
  Launch l(ctx, "widen");
  widen_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, t.stream>>>(freq.ptr, n, d_out);
  return STB_OK;
}

namespace {
// All scratch of a sort comes from one arena kept by the handle (grow-only): a sort allocates
// nothing once the handle has seen a tree of this size.
struct SortLayout {
  uint64_t arena_bytes = 0, n_max = 1;
  uint64_t max_off = 0, hist_off = 0, row_off = 0, ka_off = 0, va_off = 0, kb_off = 0, vb_off = 0;
  std::vector<uint64_t> freq_off, newpos_off;
  uint64_t carve(uint64_t bytes) {
    const uint64_t off = arena_bytes;
    arena_bytes += (bytes + 255) & ~255ull;
    return off;
  }
  explicit SortLayout(const Tree& t) {
    const size_t L = t.layers.size();
    freq_off.resize(L);
    newpos_off.resize(L);
    max_off = carve(2 * L * 4);  // per child layer: largest and smallest frequency
    for (size_t c = 0; c < L; ++c) {
      const uint64_t n = std::max<uint64_t>(child_count(t, c), 1);
      n_max = std::max(n_max, n);
      freq_off[c] = carve(n * 4);
      newpos_off[c] = carve(n * 4);
    }
    const uint64_t nblocks_max = ceil_div(n_max, RS_TILE);
    hist_off = carve(256 * nblocks_max * 4);
    row_off = carve(256 * 4);
    ka_off = carve(n_max * 4);
    va_off = carve(n_max * 4);
    kb_off = carve(n_max * 4);
    vb_off = carve(n_max * 4);
  }
};
}  // namespace

// A spare is as large as the buffer it will change places with, not as its contents: a layer's two buffers then
// have one size, and the block that the next build frees is the block that it asks for again (the stream-ordered
// pool serves it at once; with exact-size spares it had to grow by a gigabyte every other build, 0.1-0.9 s each time).
static int reserve_spares(Tree& t) {
  STB_CUDA(t, t.spare_leaves.ensure(std::max<uint64_t>(t.n_leaves, t.leaves.count), t.stream));
  if (t.spare_nodes.size() < t.layers.size()) t.spare_nodes.resize(t.layers.size());
  for (size_t k = 0; k < t.layers.size(); ++k)
    STB_CUDA(t, t.spare_nodes[k].ensure(std::max<uint64_t>(t.layers[k].count, t.layers[k].nodes.count), t.stream));
  return STB_OK;
}

int sort_reserve(Tree& t) {
  if (!t.built) return STB_OK;
  const SortLayout lay(t);
  STB_CUDA(t, t.sort_arena.ensure(lay.arena_bytes, t.stream));
  return reserve_spares(t);
}

int sort_tree(Tree& t) {
  if (!t.built) return t.fail(STB_ERR_NOT_BUILT, "sort_tree on an empty tree");
  cudaStream_t st = t.stream;
  const size_t L = t.layers.size();
  // child layer c (0 = leaves, c>0 = node layer c-1) is referenced from node layer c.
  const SortLayout lay(t);
  const std::vector<uint64_t>&freq_off = lay.freq_off, &newpos_off = lay.newpos_off;
  const uint64_t max_off = lay.max_off, hist_off = lay.hist_off, row_off = lay.row_off, ka_off = lay.ka_off, va_off = lay.va_off,
                 kb_off = lay.kb_off, vb_off = lay.vb_off;
  STB_CUDA(t, t.sort_arena.ensure(lay.arena_bytes, st));
  char* arena = t.sort_arena.ptr;
  auto words = [&](uint64_t off) { return reinterpret_cast<uint32_t*>(arena + off); };
  std::vector<uint32_t*> freq(L), newpos(L);
  uint32_t* d_max = words(max_off);
  uint32_t* d_min = d_max + L;
  STB_CUDA(t, cudaMemsetAsync(d_max, 0, L * 4, st));
  STB_CUDA(t, cudaMemsetAsync(d_min, 0xff, L * 4, st));
  for (size_t c = 0; c < L; ++c) {
    freq[c] = words(freq_off[c]);
    newpos[c] = words(newpos_off[c]);
    STB_TRY(histogram_into(t, c, freq[c]));
    const uint32_t n = (uint32_t)child_count(t, c);
    Launch l(t, "freq_max");
    const unsigned nb = (unsigned)std::min<uint64_t>(ceil_div(ceil_div(n, 4), HS_THREADS), 1184);
    max_kernel<<<nb, HS_THREADS, 0, st>>>(freq[c], n, d_max + c, d_min + c);
  }
  std::vector<uint32_t> maxf(2 * L);
  STB_CUDA(t, cudaMemcpyAsync(maxf.data(), d_max, 2 * L * 4, cudaMemcpyDeviceToHost, st));
  STB_CUDA(t, cudaStreamSynchronize(st));

  // ranks
  std::vector<bool> permuted(L, false);
  for (size_t c = 0; c < L; ++c) {
    const uint32_t n = (uint32_t)child_count(t, c);
    int passes = 0;
    const uint32_t minf = std::min(maxf[L + c], maxf[c]);
    for (uint32_t span = maxf[c] - minf; span; span >>= 8) ++passes;  // keys are maxf - freq in [0, maxf - minf]
    if (passes == 0 || n < 2) continue;  // every frequency equal: stable sort = identity
    permuted[c] = true;
    const uint32_t nblocks = (uint32_t)ceil_div(n, RS_TILE);
    uint32_t *hist = words(hist_off), *row_total = words(row_off);
    uint32_t *keys_a = words(ka_off), *vals_a = words(va_off), *keys_b = words(kb_off), *vals_b = words(vb_off);
    const uint32_t* kin = freq[c];
    const uint32_t* vin = nullptr;
    for (int p = 0; p < passes; ++p) {
      const int shift = 8 * p;
      const bool first = p == 0, last = p == passes - 1;
      uint32_t* kout = last ? nullptr : ((p & 1) ? keys_b : keys_a);
      uint32_t* vout = last ? newpos[c] : ((p & 1) ? vals_b : vals_a);
      {
        Launch l(t, "radix_hist");
        radix_hist_kernel<<<nblocks, RS_THREADS, 0, st>>>(kin, n, maxf[c], shift, nblocks, hist);
      }
      {
        Launch l(t, "radix_rowscan");  // one row per digit
        exclusive_scan_rows_kernel<<<256, 1024, 0, st>>>(hist, nblocks, row_total);
      }
      {
        Launch l(t, "radix_scatter");
        if (first && last) radix_scatter_kernel<true, true><<<nblocks, RS_THREADS, 0, st>>>(kin, vin, n, maxf[c], shift, nblocks, hist, row_total, kout, vout);
        else if (first) radix_scatter_kernel<true, false><<<nblocks, RS_THREADS, 0, st>>>(kin, vin, n, maxf[c], shift, nblocks, hist, row_total, kout, vout);
        else if (last) radix_scatter_kernel<false, true><<<nblocks, RS_THREADS, 0, st>>>(kin, vin, n, maxf[c], shift, nblocks, hist, row_total, kout, vout);
        else radix_scatter_kernel<false, false><<<nblocks, RS_THREADS, 0, st>>>(kin, vin, n, maxf[c], shift, nblocks, hist, row_total, kout, vout);
      }
      kin = kout;
      vin = vout;
    }
  }

  // apply: leaves, then every node layer (the top layer keeps its order, :455/:469).  A layer is
  // permuted into its spare, and the two buffers change roles (no copy back).
  STB_TRY(reserve_spares(t));
  if (permuted[0]) {
    {
      Launch l(t, "permute_leaves");
      permute_leaves_kernel<<<(unsigned)ceil_div(t.n_leaves, HS_THREADS), HS_THREADS, 0, st>>>(t.leaves.ptr, (uint32_t)t.n_leaves, newpos[0],
                                                                                               t.spare_leaves.ptr);
    }
    std::swap(t.leaves, t.spare_leaves);
  }
  for (size_t k = 0; k < L; ++k) {
    const uint32_t* child_map = permuted[k] ? newpos[k] : nullptr;
    const uint32_t* dst_map = (k + 1 < L && permuted[k + 1]) ? newpos[k + 1] : nullptr;
    if (!child_map && !dst_map) continue;
    const uint32_t n = (uint32_t)t.layers[k].count;
    {
      Launch l(t, "permute_rewire");
      permute_rewire_kernel<<<(unsigned)ceil_div(n, HS_THREADS), HS_THREADS, 0, st>>>(t.layers[k].nodes.ptr, n, child_map, dst_map, t.spare_nodes[k].ptr);
    }
    std::swap(t.layers[k].nodes, t.spare_nodes[k]);
  }
  t.plan_valid = false;
  STB_CUDA(t, cudaStreamSynchronize(st));
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

}  // namespace stb
