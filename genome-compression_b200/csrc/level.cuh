// level.cuh — device code shared by the level pipelines of build.cu (one GPU) and shard.cu
// (sharded): tiles of a level, first-occurrence counts, id assignment.
#pragma once

#include "common.cuh"
#include "scan.cuh"

namespace stb {

constexpr int LVL_THREADS = 256;
constexpr int LVL_ITERS = 4;
constexpr int LVL_TILE = LVL_THREADS * LVL_ITERS;  // positions per CTA in count/assign/resolve

struct LevelTable {
  Slot* slots;        // hash mode: cap + 1 slots
  uint32_t* dminpos;  // direct mode: 4^S entries each
  uint32_t* dids;
  uint32_t cap;
  uint32_t* first_bits = nullptr;  // the level's first-occurrence bitmap, kept current by the inserts
};

__device__ __forceinline__ void load_children(const uint32_t* __restrict__ cur, uint32_t n_cur, uint32_t p, uint32_t& l, uint32_t& r) {
  if (2 * (uint64_t)p + 1 < n_cur) {
    const uint2 pr = __ldg(reinterpret_cast<const uint2*>(cur) + p);
    l = pr.x;
    r = pr.y;
  } else {  // odd tail: node{last, nullptr} (utility.h:17-29)
    l = cur[2 * (uint64_t)p];
    r = PTR_NULL;
  }
}

enum { MODE_LEAF_DIRECT = 0, MODE_LEAF_HASH = 1, MODE_NODE = 2 };

// Loads the tile's 32 bitmap words (one per warp and iteration), leaves the exclusive prefix of
// their popcounts in word_pref[0..31] and the tile's total in word_pref[32].
__device__ __forceinline__ void tile_prefix(const uint32_t* __restrict__ bitmask, uint32_t block, uint32_t n, uint32_t (&words)[LVL_ITERS],
                                            uint32_t* word_pref) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int it = 0; it < LVL_ITERS; ++it) {
    const uint32_t p0 = block * LVL_TILE + it * LVL_THREADS + warp * 32;
    words[it] = p0 < n ? bitmask[p0 >> 5] : 0u;
    if (lane == 0) word_pref[it * (LVL_THREADS / 32) + warp] = __popc(words[it]);
  }
  __syncthreads();
  if (warp == 0) {
    const uint32_t v = word_pref[lane];
    const uint32_t x = warp_inclusive_sum(v);
    word_pref[lane] = x - v;
    if (lane == 31) word_pref[32] = x;
  }
  __syncthreads();
}

// The first occurrence at position p, whose id is `rank`: append its item to the layer in id order and
// emit its finished pointer.  Node items are recomputed from the child pointers (coalesced) rather than
// fetched from a table (random).
// `id_add` (sharded build): the ids of this rank's slice start there; the slice itself is stored from 0.
template <int MODE>
__device__ __forceinline__ void assign_position(uint32_t p, uint32_t rank, uint32_t* __restrict__ tmp, const LevelTable& tab, void* __restrict__ uniq,
                                                int S, const uint32_t* __restrict__ children, uint32_t n_children, uint32_t id_add = 0u) {
  const uint32_t t = MODE == MODE_NODE ? 0u : tmp[p];
  const uint32_t s = t & IDX_MASK;
  uint32_t flags = t & ~IDX_MASK;
  if (MODE == MODE_LEAF_DIRECT && (s & LEAF_SIDE)) {
    reinterpret_cast<unsigned long long*>(uniq)[rank] = __ldcg(&tab.slots[s & (LEAF_SIDE - 1u)].key);
    flags &= ~LEAF_SIDE;
  } else if (MODE == MODE_LEAF_DIRECT) {
    tab.dids[s] = rank;
    reinterpret_cast<unsigned long long*>(uniq)[rank] = leaf_from_2bit(s, S);
  } else if (MODE == MODE_LEAF_HASH) {
    reinterpret_cast<unsigned long long*>(uniq)[rank] = (s == tab.cap) ? EMPTY_KEY : __ldcg(&tab.slots[s].key);
  } else {
    uint32_t l, r, cl, cr;
    load_children(children, n_children, p, l, r);
    canonical_node(l, r, cl, cr, flags);
    reinterpret_cast<uint2*>(uniq)[rank] = make_uint2(cl, cr);
  }
  tmp[p] = finish_pointer(id_add + rank, flags);
}

// First occurrences of one tile: id = rank in position order.
template <int MODE>
__device__ __forceinline__ void assign_tile(uint32_t block, uint32_t base, const uint32_t (&words)[LVL_ITERS], const uint32_t* word_pref,
                                            uint32_t* __restrict__ tmp, uint32_t n, const LevelTable& tab, void* __restrict__ uniq, int S,
                                            const uint32_t* __restrict__ children, uint32_t n_children, uint32_t id_add = 0u) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int it = 0; it < LVL_ITERS; ++it) {
    const uint32_t p = block * LVL_TILE + it * LVL_THREADS + threadIdx.x;
    if (p < n && ((words[it] >> lane) & 1u)) {
      const uint32_t rank = base + word_pref[it * (LVL_THREADS / 32) + warp] + __popc(words[it] & ((1u << lane) - 1u));
      assign_position<MODE>(p, rank, tmp, tab, uniq, S, children, n_children, id_add);
    }
  }
}

// ids = ranks of the first occurrences in position order.  Two levels of counts instead of a scan:
// count_kernel leaves the number of first occurrences of every tile in blockcnt[] and adds it to
// its chunk's total (CHUNK_TILES tiles per chunk); a tile's base is then the sum of the chunk
// totals before its chunk plus the tile counts before it inside the chunk - at most a thousand
// L2-resident words per CTA at 3.1 Gbp, and no CTA ever waits for another one.  (A single-pass
// scan with decoupled look-back was measured here first: with 1024-position tiles the look-back
// chains through every tile in flight and the kernel was 2-4x slower than this, profiles/README.md.)
constexpr uint32_t CHUNK_TILES = 256;

// `wpref` (optional, the rank directory below): receives the exclusive prefix of the popcounts of the
// tile's 32 bitmap words, at the words' indices counted from the window's first tile.
__device__ __forceinline__ void count_tile(const uint32_t* __restrict__ bitmask, uint32_t tile, uint32_t rel, uint32_t* __restrict__ blockcnt,
                                           uint32_t* __restrict__ chunkcnt, uint16_t* __restrict__ wpref = nullptr) {
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t v = __popc(bitmask[(uint64_t)tile * (LVL_TILE / 32) + lane]);
  uint32_t c;
  if (wpref) {
    const uint32_t x = warp_inclusive_sum(v);
    wpref[(uint64_t)rel * (LVL_TILE / 32) + lane] = (uint16_t)(x - v);
    c = __shfl_sync(0xffffffffu, x, 31);
  } else {
    c = warp_sum(v);
  }
  if (lane == 0) {
    blockcnt[rel] = c;
    if (c) atomicAdd(chunkcnt + rel / CHUNK_TILES, c);
  }
}

// one warp per tile; tiles [first_block, first_block + nb) of the level, counts indexed from 0
static __global__ void __launch_bounds__(256)
count_kernel(const uint32_t* __restrict__ bitmask, uint32_t first_block, uint32_t nb, uint32_t* __restrict__ blockcnt,
             uint32_t* __restrict__ chunkcnt, uint16_t* __restrict__ wpref = nullptr) {
  const uint32_t rel = (blockIdx.x * 256 + threadIdx.x) >> 5;
  if (rel < nb) count_tile(bitmask, first_block + rel, rel, blockcnt, chunkcnt, wpref);
}

// Rank directory of a whole level (node levels of the one-shot build, DESIGN.md §4).  Once the level's
// bitmap is final, the id of any first occurrence q is
//   tilebase[q / LVL_TILE] + wpref[q / 32] + popc(bitmap[q / 32] & lanes below q % 32),
// so a later occurrence finds the id of its first occurrence without reading that position's pointer,
// and both are finished in one pass.  Bitmap (n / 8 bytes), word prefixes (n / 16 bytes; a tile holds at
// most 1024 first occurrences, 16 bits) and tile bases (n / 256 bytes) are all L2-sized.
struct RankDir {
  uint16_t* wpref;     // per bitmap word: first occurrences before it in its tile (count_kernel)
  uint32_t* tilebase;  // per tile: first occurrences before it in the level (tile_bases_kernel)
};

// One CTA of CHUNK_TILES threads per chunk of tiles: tilebase[tile] = the chunk totals before the chunk
// + the tile counts before the tile inside it.  The last CTA leaves the level's total in *total_out.
static __global__ void __launch_bounds__(CHUNK_TILES)
tile_bases_kernel(const uint32_t* __restrict__ blockcnt, const uint32_t* __restrict__ chunkcnt, uint32_t nb, uint32_t* __restrict__ tilebase,
                  uint32_t* __restrict__ total_out) {
  __shared__ uint32_t red_a[CHUNK_TILES / 32], red_b[CHUNK_TILES / 32];
  const uint32_t chunk = blockIdx.x, tile = chunk * CHUNK_TILES + threadIdx.x;
  uint32_t before = 0;
  for (uint32_t i = threadIdx.x; i < chunk; i += CHUNK_TILES) before += chunkcnt[i];
  uint32_t chunk_base, chunk_total;
  block_exclusive_sum<CHUNK_TILES>(before, red_a, &chunk_base);
  const uint32_t in_chunk = block_exclusive_sum<CHUNK_TILES>(tile < nb ? blockcnt[tile] : 0u, red_b, &chunk_total);
  if (tile < nb) tilebase[tile] = chunk_base + in_chunk;
  if (chunk == gridDim.x - 1 && threadIdx.x == 0) *total_out = chunk_base + chunk_total;
}

// Sum over the CTA of: the chunk totals before tile `rel`'s chunk + the tile counts before it in
// its chunk.  `red` is shared scratch of LVL_THREADS / 32 words; the caller synchronises before
// reading the result of the next call into the same scratch.
__device__ __forceinline__ uint32_t tile_base(uint32_t rel, const uint32_t* __restrict__ blockcnt, const uint32_t* __restrict__ chunkcnt,
                                              uint32_t* red) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t chunk = rel / CHUNK_TILES, in_chunk = chunk * CHUNK_TILES + threadIdx.x;
  uint32_t part = in_chunk < rel ? blockcnt[in_chunk] : 0u;
  for (uint32_t i = threadIdx.x; i < chunk; i += LVL_THREADS) part += chunkcnt[i];
  part = warp_sum(part);
  if (lane == 0) red[warp] = part;
  __syncthreads();
  uint32_t base = 0;
#pragma unroll
  for (int w = 0; w < LVL_THREADS / 32; ++w) base += red[w];
  return base;
}

// `carry_in` (streaming build): the level's running total before this launch's tiles; the last
// tile leaves the new total in *total_out (a different word: other CTAs still read carry_in).
template <int MODE>
__global__ void __launch_bounds__(LVL_THREADS)
assign_kernel(uint32_t* __restrict__ tmp, uint32_t n, LevelTable tab, const uint32_t* __restrict__ bitmask,
              const uint32_t* __restrict__ blockcnt, const uint32_t* __restrict__ chunkcnt, uint32_t first_block,
              const uint32_t* __restrict__ carry_in, uint32_t* __restrict__ total_out, void* __restrict__ uniq, int S,
              const uint32_t* __restrict__ children, uint32_t n_children, const uint32_t* __restrict__ id_offset = nullptr) {
  static_assert(CHUNK_TILES == LVL_THREADS, "tile_base reads one tile count per thread");
  __shared__ uint32_t word_pref[33];
  __shared__ uint32_t red[LVL_THREADS / 32];
  const uint32_t rel = blockIdx.x, block = first_block + rel;
  // a tile without first occurrences has nothing to assign (most tiles of a genome's leaf level: the 4^12
  // possible leaves have nearly all occurred after the first few per cent of the text)
  if (rel != gridDim.x - 1 && blockcnt[rel] == 0u) return;
  const uint32_t base = tile_base(rel, blockcnt, chunkcnt, red) + (carry_in ? *carry_in : 0u);
  uint32_t words[LVL_ITERS];
  tile_prefix(bitmask, block, n, words, word_pref);
  if (rel == gridDim.x - 1 && threadIdx.x == 0) *total_out = base + word_pref[32];
  assign_tile<MODE>(block, base, words, word_pref, tmp, n, tab, uniq, S, children, n_children, id_offset ? *id_offset : 0u);
}

// Leaf level of the sharded builds (shard.cu, dist.cu), where the leaf table is replicated: minpos[c] is
// the first global position of code c.  Sets the bit of every such position.  An unused entry holds
// 0xffffffff (shard.cu) or 0x7f7f7f7f (dist.cu); positions are below 2^30, so both fail the test.
static __global__ void __launch_bounds__(256)
mark_first_kernel(const uint32_t* __restrict__ minpos, uint32_t entries, uint32_t* __restrict__ bits) {
  const uint32_t c = blockIdx.x * 256 + threadIdx.x;
  if (c >= entries) return;
  const uint32_t q = __ldg(minpos + c);
  if (q < 0x7f7f7f7fu) atomicOr(bits + (q >> 5), 1u << (q & 31));
}

// ... and finishes a rank's leaf pointers from the id table: tmp[i] = code | flags, as the leaf insert left
// it.  tmp == pointers finishes them in place.
static __global__ void __launch_bounds__(256)
finish_leaves_kernel(const uint32_t* tmp, uint64_t n, const uint32_t* __restrict__ ids, uint32_t* pointers) {
  const uint64_t i = (uint64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint32_t t = tmp[i];
  pointers[i] = finish_pointer(__ldg(ids + (t & IDX_MASK)), t & ~IDX_MASK);
}

}  // namespace stb
