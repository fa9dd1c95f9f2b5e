// dist.cu — stage kernels of the multi-GPU (sharded) build; protocol in
// include/shared_tree_b200_dist.h.  Collectives are the caller's (torch.distributed / NCCL).
//
// Node ids stay first-occurrence ranks in GLOBAL position order: the owner of a key keeps
// the minimum global position, every first occurrence is one bit in a bitmap over the level's
// positions, and id(q) = number of set bits below q — a pure function of the (all-reduced)
// bitmap that every rank evaluates locally.
#include <algorithm>

#include "dist.cuh"
#include "level.cuh"
#include "scan.cuh"

namespace stb {

template <int KIND>
__global__ void __launch_bounds__(DP_THREADS)
partition_hist_kernel(const void* __restrict__ items, uint64_t n_items, uint64_t n_pos, int S, int world, uint32_t nblocks,
                      uint32_t* __restrict__ hist) {
  __shared__ uint32_t cnt[MAX_WORLD];
  if (threadIdx.x < MAX_WORLD) cnt[threadIdx.x] = 0;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31;
#pragma unroll
  for (int it = 0; it < DP_ITEMS; ++it) {
    const uint64_t i = (uint64_t)blockIdx.x * DP_TILE + it * DP_THREADS + threadIdx.x;
    uint32_t o = 0xffffffffu;
    if (i < n_pos) {
      unsigned long long key;
      uint32_t f;
      produce<KIND>(items, n_items, S, i, key, f);
      o = owner_of(key, world);
    }
    for (int w = 0; w < world; ++w) {
      const uint32_t m = __ballot_sync(0xffffffffu, o == (uint32_t)w);
      if (lane == 0 && m) atomicAdd(&cnt[w], (uint32_t)__popc(m));
    }
  }
  __syncthreads();
  if (threadIdx.x < world) hist[threadIdx.x * nblocks + blockIdx.x] = cnt[threadIdx.x];
}

template <int KIND>
__global__ void __launch_bounds__(DP_THREADS)
partition_scatter_kernel(const void* __restrict__ items, uint64_t n_items, uint64_t n_pos, int S, int world, uint64_t gpos0,
                         uint32_t nblocks, const uint32_t* __restrict__ hist, const uint32_t* __restrict__ row_total,
                         unsigned long long* __restrict__ keys, uint32_t* __restrict__ gpos, uint32_t* __restrict__ meta) {
  __shared__ uint32_t cnt[DP_ITEMS * DP_WARPS][MAX_WORLD];  // per (row, warp) counts -> offsets
  __shared__ uint32_t base[MAX_WORLD];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < MAX_WORLD) {
    uint32_t b = 0;
    for (int w = 0; w < (int)threadIdx.x && w < world; ++w) b += row_total[w];
    base[threadIdx.x] = threadIdx.x < world ? b + hist[threadIdx.x * nblocks + blockIdx.x] : 0u;
  }
  unsigned long long key[DP_ITEMS];
  uint32_t flg[DP_ITEMS], own[DP_ITEMS], rank_in_warp[DP_ITEMS];
#pragma unroll
  for (int it = 0; it < DP_ITEMS; ++it) {
    const uint64_t i = (uint64_t)blockIdx.x * DP_TILE + it * DP_THREADS + threadIdx.x;
    own[it] = 0xffffffffu;
    key[it] = 0;
    flg[it] = 0;
    rank_in_warp[it] = 0;
    if (i < n_pos) {
      produce<KIND>(items, n_items, S, i, key[it], flg[it]);
      own[it] = owner_of(key[it], world);
    }
    for (int w = 0; w < world; ++w) {
      const uint32_t m = __ballot_sync(0xffffffffu, own[it] == (uint32_t)w);
      if (own[it] == (uint32_t)w) rank_in_warp[it] = __popc(m & ((1u << lane) - 1u));
      if (lane == 0) cnt[it * DP_WARPS + warp][w] = __popc(m);
    }
  }
  __syncthreads();
  // exclusive scan over the (row, warp) sequence, per owner: index order inside the CTA
  if (threadIdx.x < world) {
    uint32_t run = base[threadIdx.x];
    for (int j = 0; j < DP_ITEMS * DP_WARPS; ++j) {
      const uint32_t c = cnt[j][threadIdx.x];
      cnt[j][threadIdx.x] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < DP_ITEMS; ++it) {
    const uint64_t i = (uint64_t)blockIdx.x * DP_TILE + it * DP_THREADS + threadIdx.x;
    if (i < n_pos) {
      const uint32_t dst = cnt[it * DP_WARPS + warp][own[it]] + rank_in_warp[it];
      keys[dst] = key[it];
      gpos[dst] = (uint32_t)(gpos0 + i);
      meta[dst] = (uint32_t)i | flg[it];
    }
  }
}

// Owner side.  The same three ideas as the single-GPU level (build.cu): a singleton filter in
// front of the table (cells are private to the owner, who sees every record of its keys), the
// first-occurrence bitmap kept by XOR toggles during the insert, and answers that touch the
// table only for the records that turned out NOT to be first occurrences.
__global__ void __launch_bounds__(256)
owner_filter_kernel(const unsigned long long* __restrict__ keys, uint32_t n, uint32_t* plane_a, uint32_t* plane_b, uint32_t log2_bits) {
  for (uint32_t j = blockIdx.x * 1024 + threadIdx.x; j < min(n, (blockIdx.x + 1) * 1024u); j += 256) {
    uint32_t word, bit;
    owner_filter_cell(__ldg(keys + j), log2_bits, word, bit);
    if (atomicOr(plane_a + word, bit) & bit) atomicOr(plane_b + word, bit);
  }
}

__global__ void __launch_bounds__(256)
owner_insert_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ gpos, uint32_t n, Slot* tab,
                    uint32_t cap, uint32_t* __restrict__ slot_of, uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ plane_b,
                    uint32_t log2_bits) {
  for (uint32_t j = blockIdx.x * 1024 + threadIdx.x; j < min(n, (blockIdx.x + 1) * 1024u); j += 256) {
    const unsigned long long key = __ldg(keys + j);
    const uint32_t pos = __ldg(gpos + j);
    if (plane_b) {
      uint32_t word, bit;
      owner_filter_cell(key, log2_bits, word, bit);
      if (!(__ldcg(plane_b + word) & bit)) {
        atomicOr(bitmap + (pos >> 5), 1u << (pos & 31));
        slot_of[j] = OWNER_SINGLETON;
        continue;
      }
    }
    slot_of[j] = table_insert<true>(tab, cap, key, pos, bitmap);
  }
}

__global__ void __launch_bounds__(256)
owner_answer_kernel(const uint32_t* __restrict__ gpos, uint32_t n, const Slot* tab, uint32_t* __restrict__ slot_then_answer,
                    const uint32_t* __restrict__ bitmap) {
  for (uint32_t j = blockIdx.x * 1024 + threadIdx.x; j < min(n, (blockIdx.x + 1) * 1024u); j += 256) {
    const uint32_t pos = __ldg(gpos + j);
    const bool first = (__ldcg(bitmap + (pos >> 5)) >> (pos & 31)) & 1u;
    slot_then_answer[j] = first ? pos : __ldcg(&tab[slot_then_answer[j]].minpos);
  }
}

// per-CTA popcount of 1024 words
__global__ void __launch_bounds__(256)
popc_blocks_kernel(const uint32_t* __restrict__ bitmap, uint64_t n_words, uint32_t* __restrict__ block_sum) {
  __shared__ uint32_t warp_totals[8];
  uint32_t c = 0;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const uint64_t w = (uint64_t)blockIdx.x * 1024 + it * 256 + threadIdx.x;
    if (w < n_words) c += __popc(bitmap[w]);
  }
  uint32_t total;
  block_exclusive_sum<256>(c, warp_totals, &total);
  if (threadIdx.x == 0) block_sum[blockIdx.x] = total;
}

// word_prefix[w] = number of set bits in words [0, w); one CTA per 1024 words (sequential in 4 rows)
__global__ void __launch_bounds__(256)
word_prefix_kernel(const uint32_t* __restrict__ bitmap, uint64_t n_words, const uint32_t* __restrict__ block_prefix,
                   uint32_t* __restrict__ word_prefix) {
  __shared__ uint32_t warp_totals[8];
  uint32_t carry = block_prefix[blockIdx.x];
  for (int it = 0; it < 4; ++it) {
    const uint64_t w = (uint64_t)blockIdx.x * 1024 + it * 256 + threadIdx.x;
    uint32_t row_total;
    const uint32_t before = block_exclusive_sum<256>(w < n_words ? __popc(bitmap[w]) : 0u, warp_totals, &row_total);
    if (w < n_words) word_prefix[w] = carry + before;
    carry += row_total;
    __syncthreads();  // the next row writes warp_totals again
  }
}

// Send order: every later occurrence gets the id of its key's first position.
__global__ void __launch_bounds__(256)
finish_rest_kernel(uint64_t n_pos, uint64_t gpos0, const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ word_prefix,
                   uint64_t n_bits, uint64_t n_words, const uint32_t* __restrict__ meta, const uint32_t* __restrict__ answers,
                   uint32_t* __restrict__ pointers) {
  const uint64_t j = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (j >= n_pos) return;
  const uint32_t m = __ldg(meta + j), q = __ldg(answers + j);
  const uint32_t pos = m & IDX_MASK;
  if ((uint64_t)q == gpos0 + pos) return;  // a first occurrence, done in position order
  pointers[pos] = finish_pointer(rank_of(bitmap, word_prefix, n_bits, n_words, q), m & ~IDX_MASK);
}

// ---- ACGT-only leaves: replicated direct-addressed table instead of the record exchange ----
constexpr uint32_t DIRECT_EMPTY = 0x7f7f7f7fu;  // > any position, positive as int32 (all-reduce MIN)

__global__ void __launch_bounds__(256)
direct_ids_kernel(const uint32_t* __restrict__ table, uint32_t entries, const uint32_t* __restrict__ bitmap,
                  const uint32_t* __restrict__ word_prefix, uint64_t n_bits, uint64_t n_words, int S, uint32_t* __restrict__ ids,
                  unsigned long long* __restrict__ leaves_out) {
  const uint32_t s = blockIdx.x * 256 + threadIdx.x;
  if (s >= entries) return;
  const uint32_t mp = __ldg(table + s);
  if (mp >= DIRECT_EMPTY) return;
  const uint32_t id = rank_of(bitmap, word_prefix, n_bits, n_words, mp);
  ids[s] = id;
  leaves_out[id] = leaf_from_2bit(s, S);
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_dist_pack_body(stb_tree* ctx, const char* body_dev, uint64_t n_leaves, uint64_t* leaves_dev) {
  if (!ctx || (!body_dev && n_leaves) || (!leaves_dev && n_leaves)) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  if (reinterpret_cast<uintptr_t>(body_dev) & 15u) return ctx->fail(STB_ERR_INVALID_ARG, "body must be 16-byte aligned");
  return pack_body(*ctx, body_dev, n_leaves, reinterpret_cast<unsigned long long*>(leaves_dev));
}

int stb_dist_partition(stb_tree* ctx, int kind, const void* items_dev, uint64_t n_items, uint64_t gpos0, int world,
                       uint64_t* keys_dev, uint32_t* gpos_dev, uint32_t* meta_dev, uint32_t* counts_dev) {
  if (!ctx || world < 1 || world > MAX_WORLD || (kind != 0 && kind != 1) || !counts_dev) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  Tree& t = *ctx;
  cudaStream_t st = t.stream;
  const uint64_t n_pos = kind == 0 ? n_items : ceil_div(n_items, 2);
  if (n_pos >= (1ull << 29)) return t.fail(STB_ERR_TOO_LARGE, "a rank holds 2^29 or more positions of one level");
  if (n_pos == 0) {
    STB_CUDA(t, cudaMemsetAsync(counts_dev, 0, world * 4, st));
    return STB_OK;
  }
  const uint32_t nblocks = (uint32_t)ceil_div(n_pos, DP_TILE);
  DevBuf<uint32_t> hist;
  STB_CUDA(t, hist.alloc((uint64_t)world * nblocks, st));
  {
    Launch l(t, "dist_partition_hist");
    if (kind == 0) partition_hist_kernel<0><<<nblocks, DP_THREADS, 0, st>>>(items_dev, n_items, n_pos, t.S, world, nblocks, hist.ptr);
    else partition_hist_kernel<1><<<nblocks, DP_THREADS, 0, st>>>(items_dev, n_items, n_pos, t.S, world, nblocks, hist.ptr);
  }
  {
    Launch l(t, "dist_rowscan");
    exclusive_scan_rows_kernel<<<world, 1024, 0, st>>>(hist.ptr, nblocks, counts_dev);  // one row per owner
  }
  {
    Launch l(t, "dist_partition_scatter");
    if (kind == 0)
      partition_scatter_kernel<0><<<nblocks, DP_THREADS, 0, st>>>(items_dev, n_items, n_pos, t.S, world, gpos0, nblocks, hist.ptr, counts_dev,
                                                                  reinterpret_cast<unsigned long long*>(keys_dev), gpos_dev, meta_dev);
    else
      partition_scatter_kernel<1><<<nblocks, DP_THREADS, 0, st>>>(items_dev, n_items, n_pos, t.S, world, gpos0, nblocks, hist.ptr, counts_dev,
                                                                  reinterpret_cast<unsigned long long*>(keys_dev), gpos_dev, meta_dev);
  }
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

int stb_dist_owner(stb_tree* ctx, const uint64_t* keys_dev, const uint32_t* gpos_dev, uint64_t n_records, void* table_dev,
                   uint32_t cap, uint32_t* answers_dev, uint32_t* bitmap_dev) {
  if (!ctx || !table_dev || cap < 2 * n_records || cap > 0x1ffffffeu) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  if (n_records == 0) return STB_OK;
  Tree& t = *ctx;
  cudaStream_t st = t.stream;
  {
    Launch l(t, "table_clear", false);
    STB_CUDA(t, cudaMemsetAsync(table_dev, 0xff, ((uint64_t)cap + 1) * sizeof(Slot), st));
  }
  // singleton filter: two bit planes of 2^k bits, k up to 28 (2 x 32 MiB: L2-resident)
  uint32_t log2_bits = 0;
  DevBuf<uint32_t> planes;
  if (n_records >= (1u << 16)) {
    log2_bits = 22;
    while (log2_bits < 28 && (1ull << log2_bits) < 2 * n_records) ++log2_bits;
    const uint64_t words = (1ull << log2_bits) / 32;
    STB_CUDA(t, planes.alloc(2 * words, st));
    STB_CUDA(t, cudaMemsetAsync(planes.ptr, 0, 2 * words * 4, st));
  }
  uint32_t* plane_a = planes.ptr;
  uint32_t* plane_b = planes.ptr ? planes.ptr + (1ull << log2_bits) / 32 : nullptr;
  const unsigned nb = (unsigned)ceil_div(n_records, 1024);
  if (plane_b) {
    Launch l(t, "dist_owner_filter");
    owner_filter_kernel<<<nb, 256, 0, st>>>(reinterpret_cast<const unsigned long long*>(keys_dev), (uint32_t)n_records, plane_a, plane_b, log2_bits);
  }
  {
    Launch l(t, "dist_owner_insert");
    owner_insert_kernel<<<nb, 256, 0, st>>>(reinterpret_cast<const unsigned long long*>(keys_dev), gpos_dev, (uint32_t)n_records,
                                            reinterpret_cast<Slot*>(table_dev), cap, answers_dev, bitmap_dev, plane_b, log2_bits);
  }
  {
    Launch l(t, "dist_owner_answer");
    owner_answer_kernel<<<nb, 256, 0, st>>>(gpos_dev, (uint32_t)n_records, reinterpret_cast<const Slot*>(table_dev), answers_dev, bitmap_dev);
  }
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

int stb_dist_rank_index(stb_tree* ctx, const uint32_t* bitmap_dev, uint64_t n_words, uint32_t* word_prefix_dev,
                        uint32_t* scratch_dev) {
  if (!ctx || !bitmap_dev || !word_prefix_dev || !scratch_dev) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  Tree& t = *ctx;
  cudaStream_t st = t.stream;
  const uint32_t nblocks = (uint32_t)ceil_div(n_words, 1024);
  {
    Launch l(t, "dist_popc_blocks");
    popc_blocks_kernel<<<nblocks, 256, 0, st>>>(bitmap_dev, n_words, scratch_dev);
  }
  {
    Launch l(t, "dist_scan");
    exclusive_scan_rows_kernel<<<1, 1024, 0, st>>>(scratch_dev, nblocks, word_prefix_dev + n_words);
  }
  {
    Launch l(t, "dist_word_prefix");
    word_prefix_kernel<<<nblocks, 256, 0, st>>>(bitmap_dev, n_words, scratch_dev, word_prefix_dev);
  }
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

int stb_dist_finish(stb_tree* ctx, int kind, const void* items_dev, uint64_t n_items, uint64_t gpos0,
                    const uint32_t* bitmap_dev, const uint32_t* word_prefix_dev, uint64_t n_level_positions,
                    const uint32_t* meta_dev, const uint32_t* answers_dev, uint32_t* pointers_dev, void* layer_slice_dev,
                    uint32_t* base_count_dev) {
  if (!ctx || (kind != 0 && kind != 1) || !bitmap_dev || !word_prefix_dev || !base_count_dev) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  Tree& t = *ctx;
  cudaStream_t st = t.stream;
  const uint64_t n_pos = kind == 0 ? n_items : ceil_div(n_items, 2);
  STB_TRY(finish_first(t, kind, items_dev, n_items, gpos0, bitmap_dev, word_prefix_dev, n_level_positions, pointers_dev, layer_slice_dev,
                       base_count_dev));
  if (n_pos) {
    const uint64_t n_words = ceil_div(n_level_positions, 32);
    Launch l(t, "dist_finish_rest");
    finish_rest_kernel<<<(unsigned)ceil_div(n_pos, 256), 256, 0, st>>>(n_pos, gpos0, bitmap_dev, word_prefix_dev, n_level_positions, n_words,
                                                                       meta_dev, answers_dev, pointers_dev);
  }
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

int stb_dist_leaf_direct_minpos(stb_tree* ctx, const char* body_dev, uint64_t n_local, uint64_t gpos0, uint32_t* table_dev,
                                uint32_t* tmp_dev, int* non_acgt) {
  if (!ctx || !table_dev || !non_acgt || (n_local && (!body_dev || !tmp_dev))) return STB_ERR_INVALID_ARG;
  if (ctx->S > 12) return ctx->fail(STB_ERR_INVALID_ARG, "direct leaf table needs dna_size <= 12");
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  if (reinterpret_cast<uintptr_t>(body_dev) & 15u) return ctx->fail(STB_ERR_INVALID_ARG, "body must be 16-byte aligned");
  if (gpos0 + n_local >= DIRECT_EMPTY) return ctx->fail(STB_ERR_TOO_LARGE, "more than 2^31 leaf positions");
  return dist_leaf_direct_minpos(*ctx, body_dev, n_local, gpos0, table_dev, tmp_dev, non_acgt);
}

int stb_dist_leaf_direct_finish(stb_tree* ctx, const uint32_t* table_dev, uint64_t n_level_positions, const uint32_t* tmp_dev,
                                uint64_t n_local, uint32_t* bitmap_dev, uint32_t* word_prefix_dev, uint32_t* scratch_dev,
                                uint32_t* ids_dev, uint32_t* pointers_dev, uint64_t* leaves_out_dev) {
  if (!ctx || !table_dev || !bitmap_dev || !word_prefix_dev || !scratch_dev || !ids_dev || !leaves_out_dev) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(ctx->device) != cudaSuccess) return STB_ERR_CUDA;
  Tree& t = *ctx;
  cudaStream_t st = t.stream;
  const uint32_t entries = 1u << (2 * t.S);
  const uint64_t n_words = ceil_div(n_level_positions, 32);
  {
    Launch l(t, "dist_direct_mark");
    mark_first_kernel<<<(unsigned)ceil_div(entries, 256), 256, 0, st>>>(table_dev, entries, bitmap_dev);
  }
  STB_TRY(stb_dist_rank_index(ctx, bitmap_dev, n_words, word_prefix_dev, scratch_dev));
  {
    Launch l(t, "dist_direct_ids");
    direct_ids_kernel<<<(unsigned)ceil_div(entries, 256), 256, 0, st>>>(table_dev, entries, bitmap_dev, word_prefix_dev, n_level_positions, n_words,
                                                                        t.S, ids_dev, reinterpret_cast<unsigned long long*>(leaves_out_dev));
  }
  if (n_local) {
    Launch l(t, "dist_direct_resolve");
    finish_leaves_kernel<<<(unsigned)ceil_div(n_local, 256), 256, 0, st>>>(tmp_dev, n_local, ids_dev, pointers_dev);
  }
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

int stb_dist_upper_levels(stb_tree* tree, const uint32_t* pointers_dev, uint64_t n_pointers, int leaf_pointers) {
  if (!tree || !pointers_dev) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(tree->device) != cudaSuccess) return STB_ERR_CUDA;
  return build_upper_levels(*tree, pointers_dev, n_pointers, leaf_pointers != 0);
}

int stb_assemble(stb_tree* tree, const uint64_t* leaves_dev, uint64_t n_leaves, uint64_t n_layers,
                 const uint64_t* layer_counts, const void* const* layers_dev, uint32_t root, uint64_t width) {
  if (!tree || !layer_counts || !layers_dev || n_layers == 0 || n_layers > 40) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(tree->device) != cudaSuccess) return STB_ERR_CUDA;
  Tree& t = *tree;
  t.clear();
  cudaStream_t st = t.stream;
  STB_CUDA(t, t.leaves.alloc(n_leaves, st));
  if (n_leaves) STB_CUDA(t, cudaMemcpyAsync(t.leaves.ptr, leaves_dev, n_leaves * 8, cudaMemcpyDeviceToDevice, st));
  for (uint64_t k = 0; k < n_layers; ++k) {
    t.layers.emplace_back();
    Layer& layer = t.layers.back();
    layer.count = layer_counts[k];
    STB_CUDA(t, layer.nodes.alloc(layer.count, st));
    if (layer.count) STB_CUDA(t, cudaMemcpyAsync(layer.nodes.ptr, layers_dev[k], layer.count * sizeof(uint2), cudaMemcpyDeviceToDevice, st));
  }
  STB_CUDA(t, cudaStreamSynchronize(st));
  t.n_leaves = n_leaves;
  t.root = root;
  t.width = width;
  t.built = true;
  t.plan_valid = false;
  return STB_OK;
}

}  // extern "C"
