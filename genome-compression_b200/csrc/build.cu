// build.cu — level-by-level bottom-up construction of the shared tree (hash-consing).
//
// Replaces tree_constructor (reference include/shared_tree.h:245-316,
// src/shared_tree.cpp:621-763) and the phmap dedup behind it.  The reference
// streams 2^22-leaf segments through per-layer hash maps, one element at a time;
// because its segments are powers of two that is equivalent to ONE global pass per
// level (SURVEY §8 a10), which is what runs here:
//
//   per level (leaves, then node layers bottom-up):
//     insert   every position canonicalises its item and lowers the item's
//              min-position in an open-addressing table (or a direct-addressed
//              table for ACGT-only leaves); whoever becomes a key's minimum
//              toggles its own bit in the level's bitmap and the bit of the
//              position it displaced (XOR commutes), so when the kernel ends the
//              bitmap marks exactly the first occurrences      [random HBM/L2]
//     scan     per-CTA popcounts of the bitmap, exclusive scan [tiny]
//     assign   first occurrences get id = rank, append the item to the layer in id
//              order and emit their pointer                    [coalesced]
//     resolve  later occurrences: slot -> min-position -> the first occurrence's
//              finished pointer -> id                          [random reads]
//
//   node levels built one kernel at a time (option fused_resolve, default on):
//     count        tile popcounts + each bitmap word's prefix inside its tile
//     tile_bases   absolute first-occurrence count before every tile
//     assign_resolve  first occurrences as in assign; a later occurrence takes the
//              rank of its first occurrence from that rank directory (bitmap, word
//              prefixes, tile bases: L2-sized), so no second pass reads the
//              first occurrence's pointer                      [coalesced + L2]
//
// IDs are first-occurrence ranks in position order, independent of which thread won
// which atomic, so the result equals the reference's sequential emplace order.
#include <cooperative_groups.h>

#include <algorithm>
#include <vector>

#include "bucket.cuh"
#include "level.cuh"
#include "pack.cuh"
#include "tree.h"

namespace stb {

struct BuildFlags {
  unsigned long long bad_symbol;  // (byte offset << 8) | upper-cased byte; ~0 = none
  uint32_t non_acgt;              // direct leaf mode cannot hold this input's leaves (no side table, or it filled up)
  uint32_t bad_leaf;              // packed input leaf with bits >= 4S
  uint32_t side_claims;           // distinct leaves in the side table
  uint32_t pad;
};

// Leaves with symbols outside ACGT (N runs, IUPAC codes) next to a direct-addressed ACGT table: they
// go to a small hash table (the level's `slots` / `cap` in direct mode) keyed by the canonical
// 4-bit word.  Real genomes have few distinct ones (all-N, and what borders on an N run), so the
// table is small; an input with more distinct such leaves than it holds raises non_acgt and the
// host rebuilds with the hash-table leaf level.  Returns the slot, or ~0 when it gave up.
__device__ __forceinline__ uint32_t side_insert(const LevelTable& tab, unsigned long long key, uint32_t pos, BuildFlags* flags) {
  if (tab.cap == 0u || *reinterpret_cast<volatile uint32_t*>(&flags->side_claims) > tab.cap / 2u) {
    flags->non_acgt = 1u;
    return 0xffffffffu;
  }
  uint32_t s = __umulhi(hash64(key), tab.cap);
  for (uint32_t steps = 0; steps < 8192u; ++steps) {
    unsigned long long k;
    uint32_t mp;
    load_slot(tab.slots + s, k, mp);
    if (k == EMPTY_KEY) {
      claim_slot(tab.slots + s, key, pos, k, mp);
      if (k == EMPTY_KEY) {  // claimed: key and min-position written together
        atomicAdd(&flags->side_claims, 1u);
        if (tab.first_bits) toggle_bit(tab.first_bits, pos);
        return s;
      }
    }
    if (k == key) {
      if (mp > pos) {
        const uint32_t old = atomicMin(&tab.slots[s].minpos, pos);
        if (tab.first_bits && old > pos) {
          toggle_bit(tab.first_bits, pos);
          toggle_bit(tab.first_bits, old);
        }
      }
      return s;
    }
    if (++s == tab.cap) s = 0;
  }
  flags->non_acgt = 1u;
  return 0xffffffffu;
}

template <bool DIRECT>
__device__ __forceinline__ void insert_leaf(unsigned long long v, int S, uint32_t pos, const LevelTable& tab,
                                            uint32_t* __restrict__ tmp_at_pos, BuildFlags* flags) {
  uint32_t f;
  const unsigned long long canon = canonical_leaf(v, S, f);
  uint32_t s;
  if (DIRECT) {
    if (!leaf_is_acgt(v, S)) {
      const uint32_t side = side_insert(tab, canon, pos, flags);
      *tmp_at_pos = side == 0xffffffffu ? 0u : (LEAF_SIDE | side | f);
      return;
    }
    s = leaf_to_2bit(canon);
    if (__ldcg(tab.dminpos + s) > pos) {
      const uint32_t old = atomicMin(tab.dminpos + s, pos);
      if (tab.first_bits && old > pos) {  // see toggle_bit (common.cuh)
        toggle_bit(tab.first_bits, pos);
        if (old != 0xffffffffu) toggle_bit(tab.first_bits, old);
      }
    }
  } else {
    s = table_insert<true>(tab.slots, tab.cap, canon, pos, tab.first_bits);
  }
  *tmp_at_pos = s | f;
}

// Leaves straight from the ASCII body: pack (dna.cpp:79-84) + canonical (dna.cpp:135)
// + emplace_leaf (shared_tree.cpp:630) fused; the packed leaves never touch HBM.
template <int S_T, bool DIRECT>
__global__ void __launch_bounds__(PACK_THREADS)
leaf_insert_text_kernel(const char* __restrict__ body, uint64_t n_leaves, int S_rt, LevelTable tab,
                        uint32_t* __restrict__ tmp, BuildFlags* flags, uint32_t pos0) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t* lut = smem;
  uint8_t* tile = smem + 256;
  const int S = S_T > 0 ? S_T : S_rt;
  const uint64_t tile_first = (uint64_t)blockIdx.x * PACK_TILE_LEAVES;
  const uint32_t here = (uint32_t)min((uint64_t)PACK_TILE_LEAVES, n_leaves - tile_first);
  stage_text_tile(lut, tile, body + tile_first * S, here * (uint32_t)S);
#pragma unroll
  for (int it = 0; it < PACK_LEAVES_PER_THREAD; ++it) {
    const uint32_t j = it * PACK_THREADS + threadIdx.x;
    if (j < here) {
      uint32_t bad = 0xFFFFFFFFu;
      const unsigned long long v = pack_leaf<S_T>(lut, tile, j, S, bad);
      if (bad != 0xFFFFFFFFu) {
        uint32_t c = tile[bad];
        if (c >= 'a' && c <= 'z') c -= 32;
        // `body` starts at leaf pos0 of the text: offsets count from the text's start, so that the smallest one is
        // the first bad byte even when the text is inserted in several launches (the streaming build)
        atomicMin(&flags->bad_symbol, (((uint64_t)pos0 * S + tile_first * S + bad) << 8) | c);
      }
      insert_leaf<DIRECT>(v, S, pos0 + (uint32_t)(tile_first + j), tab, tmp + tile_first + j, flags);
    }
  }
}

// ACGT fast path for the default leaf length (12): the whole leaf level in 32-bit registers.
// Four text bytes -> four 2-bit codes by SWAR (A0 C1 G2 T3; any other byte, in either case,
// fails the check), twelve of them = one 24-bit word whose numeric order equals the order of
// the reference's 4-bit words (A1<C2<G4<T8, same nucleotide significance), so the canonical
// variant (dna.cpp:135-143) is the minimum of {c, ~c, reverse(c), reverse(~c)} taken on that
// word, and the word itself is the direct-table index.  Anything that is not pure ACGT raises
// the non_acgt flag and the host re-runs the level through the general kernel.
__device__ __forceinline__ bool acgt_word_to_2bit(uint32_t w, uint32_t& out8) {
  const uint32_t u = w & 0xDFDFDFDFu;                       // fold case
  const uint32_t x = (u >> 1) & 0x03030303u;                // A0 C1 G3 T2
  const uint32_t idx = x ^ ((x >> 1) & 0x01010101u);        // A0 C1 G2 T3
  const uint32_t b0 = idx & 0x01010101u, b1 = (idx >> 1) & 0x01010101u, bb = b0 & b1;
  // the byte each code must have come from: 'A' + {0, 2, 6, 0x13}
  const uint32_t expect = 0x41414141u + (b0 << 1) + (b1 << 1) + (b1 << 2) + bb + (bb << 1) + (bb << 3);
  out8 = (idx * 0x01041040u) >> 24;                          // 4 codes -> 8 bits, first char lowest
  return expect == u;
}

__device__ __forceinline__ uint32_t reverse_2bit_24(uint32_t c) {
  const uint32_t r = __brev(c) >> 8;  // reverses the pairs and the bits inside each pair
  return ((r & 0x555555u) << 1) | ((r >> 1) & 0x555555u);
}

// LOOKUP (one-shot build, the leaves after a prefix whose ids are already assigned): a leaf whose code
// has an id in tab.dids is a later occurrence of a prefix leaf; it gets its finished pointer here and
// its bit in done_bits (indexed by position; a warp covers one word), and skips the min-position
// table.  Every other leaf takes the insert below and stays pending.
template <bool LOOKUP>
__device__ __forceinline__ bool acgt12_leaf(const uint8_t* smem, const uint8_t* tile, uint32_t j, uint64_t tile_first, const LevelTable& tab,
                                            uint32_t* __restrict__ tmp, BuildFlags* flags, uint32_t pos0) {
  const uint32_t* words = reinterpret_cast<const uint32_t*>(tile);
  uint32_t c0, c1, c2;
  const bool ok = acgt_word_to_2bit(words[3 * j], c0) & acgt_word_to_2bit(words[3 * j + 1], c1) & acgt_word_to_2bit(words[3 * j + 2], c2);
  if (!ok) {  // a symbol outside ACGT: the general 4-bit pack of this one leaf, into the side table
    uint32_t bad = 0xFFFFFFFFu, f4;
    const unsigned long long v = pack_leaf<12>(smem, tile, j, 12, bad);
    if (bad != 0xFFFFFFFFu) {
      uint32_t ch = tile[bad];
      if (ch >= 'a' && ch <= 'z') ch -= 32;
      // (every launch starts at leaf pos0 of the text: a lookup launch, and every chunk of the streaming build;
      // offsets count from the text's start)
      const uint64_t text0 = (uint64_t)pos0 * 12;
      atomicMin(&flags->bad_symbol, ((text0 + tile_first * 12 + bad) << 8) | ch);
    }
    const unsigned long long canon = canonical_leaf(v, 12, f4);
    const uint32_t side = side_insert(tab, canon, pos0 + (uint32_t)(tile_first + j), flags);
    tmp[tile_first + j] = side == 0xffffffffu ? 0u : (LEAF_SIDE | side | f4);
    return false;
  }
  const uint32_t c = c0 | (c1 << 8) | (c2 << 16);
  const uint32_t t = ~c & 0xFFFFFFu, m = reverse_2bit_24(c), i = ~m & 0xFFFFFFu;
  uint32_t best = c, f = 0;
  if (t < best) { best = t; f = TRANSPOSE; }
  if (m < best) { best = m; f = MIRROR; }
  if (i < best) { best = i; f = MIRROR | TRANSPOSE; }
  if (c == m) f |= INVARIANT;
  if (LOOKUP) {
    const uint32_t id = __ldcg(tab.dids + best);
    if (id != 0xffffffffu) {
      tmp[tile_first + j] = finish_pointer(id, f);
      return true;
    }
  }
  const uint32_t pos = pos0 + (uint32_t)(tile_first + j);
  if (__ldcg(tab.dminpos + best) > pos) {
    const uint32_t old = atomicMin(tab.dminpos + best, pos);
    if (tab.first_bits && old > pos) {
      toggle_bit(tab.first_bits, pos);
      if (old != 0xffffffffu) toggle_bit(tab.first_bits, old);
    }
  }
  tmp[tile_first + j] = best | f;
  return false;
}

template <bool LOOKUP>
__global__ void __launch_bounds__(PACK_THREADS)
leaf_insert_acgt12_kernel(const char* __restrict__ body, uint64_t n_leaves, LevelTable tab, uint32_t* __restrict__ tmp,
                          BuildFlags* flags, uint32_t pos0, uint32_t* __restrict__ done_bits) {
  extern __shared__ __align__(16) uint8_t smem[];
  uint8_t* tile = smem + 256;  // same layout as the general kernel (the table area is unused here)
  const uint64_t tile_first = (uint64_t)blockIdx.x * PACK_TILE_LEAVES;
  const uint32_t here = (uint32_t)min((uint64_t)PACK_TILE_LEAVES, n_leaves - tile_first);
  stage_text_tile(smem, tile, body + tile_first * 12, here * 12u);
#pragma unroll
  for (int it = 0; it < PACK_LEAVES_PER_THREAD; ++it) {
    const uint32_t j = it * PACK_THREADS + threadIdx.x;
    const bool done = j < here && acgt12_leaf<LOOKUP>(smem, tile, j, tile_first, tab, tmp, flags, pos0);
    if (LOOKUP) {  // pos0 is a multiple of 32: the warp's 32 positions are one word, lane 0 stores it whole
      const uint32_t word = __ballot_sync(0xffffffffu, done);
      if ((threadIdx.x & 31) == 0 && j < here) done_bits[(pos0 + (uint32_t)(tile_first + j)) >> 5] = word;
    }
  }
}

// Leaves from a packed array (the std::vector<dna> constructor, shared_tree.cpp:212).
template <bool DIRECT>
__global__ void __launch_bounds__(LVL_THREADS)
leaf_insert_u64_kernel(const unsigned long long* __restrict__ leaves, uint32_t n, int S, LevelTable tab,
                       uint32_t* __restrict__ tmp, BuildFlags* flags) {
  const uint32_t p = blockIdx.x * LVL_THREADS + threadIdx.x;
  if (p >= n) return;
  const unsigned long long v = __ldg(leaves + p);
  if (v & ~leaf_mask(S)) flags->bad_leaf = 1u;
  insert_leaf<DIRECT>(v, S, p, tab, tmp + p, flags);
}

// Exact singleton filter (node levels above the first).  A node can only repeat an earlier node
// if BOTH its children repeat: equal keys mean equal child ids, so the children of the later
// node are later occurrences of the children of the earlier one, and the children of the earlier
// one are first occurrences that occur again.  The child level left two bitmaps: `first` (its
// first occurrences) and `multi` (first occurrences whose key occurred again).  A position with a
// child that is a first occurrence and never occurred again holds the only node with that child:
// it is a first occurrence that nobody will ever look up, and it skips the table altogether.
// (A null right child counts as repeating: bits past the end of the child level are zero in `first`.)
__device__ __forceinline__ bool children_both_repeat(const uint32_t* __restrict__ child_first, const uint32_t* __restrict__ child_multi,
                                                     uint32_t p) {
  const uint32_t w = p >> 4, sh = (2u * p) & 31u;
  const uint32_t repeats = ~__ldg(child_first + w) | __ldg(child_multi + w);
  return ((repeats >> sh) & 3u) == 3u;
}

__device__ __forceinline__ uint32_t node_slot_start(const LevelTable& tab, uint32_t cl, uint32_t cr, uint32_t hashed,
                                                    const uint32_t* __restrict__ child_unique, uint32_t& limit) {
  limit = 0xffffffffu;
  if (!child_unique) return hashed;
  // Locality placement (node layers above the first): child ids are first-occurrence ranks, so
  // they grow with the position; a slot proportional to a child id makes neighbouring positions
  // probe neighbouring slots (one 128-byte line serves several positions instead of one line
  // per position).  Crowded neighbourhoods (one child with many partners) fall back to the hash.
  const uint32_t child = ptr_is_null(cl) ? (cr & IDX_MASK) : (cl & IDX_MASK);
  // (any deterministic function of the key will do: single-precision scaling, no 64-bit divide)
  const float ratio = __fdividef((float)tab.cap, (float)max(1u, __ldg(child_unique)));
  limit = 24u;
  // clamped in integers: (float)(cap - 9) rounds up for caps >= 2^25 and would let the probe
  // start at or past `cap`, which tagged_insert only wraps at exactly
  return min(tab.cap - 9u, (uint32_t)min(4.0e9f, (float)child * ratio)) + (hashed & 7u);
}

// One position of a node level: reduce_nodes + emplace_node (shared_tree.cpp:697-712, :662-672).
// Returns true when the position skipped the table (certified singleton).
__device__ __forceinline__ bool node_insert_position(const uint32_t* __restrict__ cur, uint32_t n_cur, uint32_t p, const LevelTable& tab,
                                                     uint32_t* __restrict__ aux, const uint32_t* __restrict__ child_unique, uint32_t serial,
                                                     const uint32_t* __restrict__ child_first, const uint32_t* __restrict__ child_multi) {
  if (child_first && !children_both_repeat(child_first, child_multi, p)) return true;  // assign recomputes the node
  uint32_t l, r, cl, cr, f, limit;
  load_children(cur, n_cur, p, l, r);
  canonical_node(l, r, cl, cr, f);
  const unsigned long long key = ((unsigned long long)cl << 32) | cr;
  const uint32_t hashed = __umulhi(hash64(key), tab.cap);
  const uint32_t start = node_slot_start(tab, cl, cr, hashed, child_unique, limit);
  aux[p] = tagged_insert(tab.slots, tab.cap, key, p, serial, start, hashed, limit, tab.first_bits) | f;
  return false;
}

__global__ void __launch_bounds__(LVL_THREADS)
node_insert_kernel(const uint32_t* __restrict__ cur, uint32_t n_cur, uint32_t n_next, LevelTable tab, uint32_t* __restrict__ aux,
                   const uint32_t* __restrict__ child_unique, uint32_t serial, const uint32_t* __restrict__ child_first,
                   const uint32_t* __restrict__ child_multi, uint32_t first_block, const uint32_t* __restrict__ enable) {
  if (enable && !*enable) return;  // the fallback of the on-chip path: runs only when a bucket overflowed
  // several positions per thread: CTAs that live for one probe each are dispatch-bound; the
  // fallback is launched with a grid that fits the machine and walks the tiles
  const uint32_t tiles = (n_next + LVL_TILE - 1) / LVL_TILE;
  for (uint32_t tile = first_block + blockIdx.x; tile < tiles; tile += gridDim.x) {
#pragma unroll 1
    for (int it = 0; it < LVL_ITERS; ++it) {
      const uint32_t p = tile * LVL_TILE + it * LVL_THREADS + threadIdx.x;
      const bool skipped = p < n_next && node_insert_position(cur, n_cur, p, tab, aux, child_unique, serial, child_first, child_multi);
      // a warp covers one word of the bitmap: certified singletons are marked with one atomic
      const uint32_t word = __ballot_sync(0xffffffffu, skipped);
      if ((threadIdx.x & 31) == 0 && word) atomicOr(tab.first_bits + (p >> 5), word);
    }
  }
}

// Later occurrences.  RESOLVE_DIRECT (ACGT leaves): the id is in the (L2-sized) id table.
// Otherwise the id is read from the finished pointer of the first occurrence, whose position is
// either in the slot aux[p] names (hash-table levels) or in aux[p] itself (levels deduplicated on
// chip, bucket.cu: `firstpos_unless` points at their overflow flag).  Hash-table levels also mark
// the first occurrence in `multi_bits`: its key occurred again (children_both_repeat reads it).
enum { RESOLVE_DIRECT = 0, RESOLVE_TABLE = 1 };
template <int MODE>
__global__ void __launch_bounds__(LVL_THREADS)
resolve_kernel(const uint32_t* aux, uint32_t* out, uint32_t n, LevelTable tab, const uint32_t* __restrict__ bitmask,
               uint32_t first_block, uint32_t* __restrict__ multi_bits, const uint32_t* __restrict__ firstpos_unless) {
  const uint32_t lane = threadIdx.x & 31;
  const bool firstpos = firstpos_unless && *firstpos_unless == 0u;
#pragma unroll
  for (int it = 0; it < LVL_ITERS; ++it) {
    const uint32_t p = (first_block + blockIdx.x) * LVL_TILE + it * LVL_THREADS + threadIdx.x;
    if (p < n) {
      const uint32_t word = bitmask[p >> 5];
      if (!((word >> lane) & 1u)) {
        const uint32_t t = aux[p];
        const uint32_t s = t & IDX_MASK;
        uint32_t id;
        if (MODE == RESOLVE_DIRECT && !(s & LEAF_SIDE)) {
          id = __ldcg(tab.dids + s);
        } else if (MODE == RESOLVE_DIRECT) {  // a side-table leaf: its first occurrence's finished pointer has the id
          id = __ldcg(out + __ldcg(&tab.slots[s & (LEAF_SIDE - 1u)].minpos)) & IDX_MASK;
        } else {
          uint32_t q = s;
          if (!firstpos) {
            q = __ldcg(&tab.slots[s].minpos);
            // test before set: the positions of an N run (or of any long run) all name the same first occurrence
            if (multi_bits && !((__ldcg(multi_bits + (q >> 5)) >> (q & 31u)) & 1u)) atomicOr(multi_bits + (q >> 5), 1u << (q & 31));
          } else if (p - q < COLLAPSE_WINDOW && !((__ldcg(bitmask + (q >> 5)) >> (q & 31u)) & 1u)) {
            // p repeats its predecessor and q is the head of its run (bucket.cu), itself a later occurrence
            q = __ldcg(aux + q) & IDX_MASK;
          }
          id = __ldcg(out + q) & IDX_MASK;
        }
        out[p] = finish_pointer(id, t & ~IDX_MASK);
      }
    }
  }
}

// A node level with its rank directory (RankDir, level.cuh) in one pass: first occurrences as in
// assign_tile, later occurrences as in resolve_kernel<RESOLVE_TABLE>, except that the id of the first
// occurrence q is q's rank, not read from out[q] - so nothing here reads a pointer this launch writes.
// Bitmap words, word prefixes and tile bases are read-only for the whole launch (ld.global.nc).
__global__ void __launch_bounds__(LVL_THREADS)
assign_resolve_kernel(const uint32_t* __restrict__ aux, uint32_t* __restrict__ out, uint32_t n, LevelTable tab, const uint32_t* __restrict__ bitmask,
                      RankDir dir, uint32_t* __restrict__ multi_bits, const uint32_t* __restrict__ firstpos_unless, void* __restrict__ uniq,
                      const uint32_t* __restrict__ children, uint32_t n_children) {
  const uint32_t lane = threadIdx.x & 31;
  const bool firstpos = firstpos_unless && *firstpos_unless == 0u;
  const uint32_t base = __ldg(dir.tilebase + blockIdx.x);
#pragma unroll
  for (int it = 0; it < LVL_ITERS; ++it) {
    const uint32_t p = blockIdx.x * LVL_TILE + it * LVL_THREADS + threadIdx.x;
    if (p >= n) continue;
    const uint32_t word = __ldg(bitmask + (p >> 5));
    if ((word >> lane) & 1u) {
      const uint32_t rank = base + __ldg(dir.wpref + (p >> 5)) + __popc(word & ((1u << lane) - 1u));
      assign_position<MODE_NODE>(p, rank, out, tab, uniq, 0, children, n_children);
      continue;
    }
    const uint32_t t = aux[p];
    uint32_t q = t & IDX_MASK;
    if (!firstpos) {
      q = __ldcg(&tab.slots[q].minpos);
      // test before set: the positions of an N run (or of any long run) all name the same first occurrence
      if (multi_bits && !((__ldcg(multi_bits + (q >> 5)) >> (q & 31u)) & 1u)) atomicOr(multi_bits + (q >> 5), 1u << (q & 31));
    }
    uint32_t qword = __ldg(bitmask + (q >> 5));
    if (firstpos && p - q < COLLAPSE_WINDOW && !((qword >> (q & 31u)) & 1u)) {
      // p repeats its predecessor and q is the head of its run (bucket.cu), itself a later occurrence
      q = __ldcg(aux + q) & IDX_MASK;
      qword = __ldg(bitmask + (q >> 5));
    }
    const uint32_t id = __ldg(dir.tilebase + q / LVL_TILE) + __ldg(dir.wpref + (q >> 5)) + __popc(qword & ((1u << (q & 31u)) - 1u));
    out[p] = finish_pointer(id, t & ~IDX_MASK);
  }
}

// Clears the level's bitmaps when the on-chip path gave up (the hash-table fallback starts from zero).
__global__ void __launch_bounds__(256) bitmaps_reset_kernel(uint32_t* __restrict__ a, uint32_t* __restrict__ b, uint32_t words,
                                                            const uint32_t* __restrict__ enable) {
  if (!*enable) return;
  for (uint32_t i = blockIdx.x * 256 + threadIdx.x; i < words; i += gridDim.x * 256) {
    a[i] = 0u;
    b[i] = 0u;
  }
}

// ---- the small top of the tree in ONE launch ----------------------------------------------
// Once a level has at most SMALL_MAX pointers, every remaining level (about a dozen) runs inside
// a single CTA: pointers ping-pong in shared memory, the hash table lives in shared memory, and
// __syncthreads() replaces the launches per level of the general path.
constexpr uint32_t SMALL_MAX = 2048;        // pointers entering the kernel (<= 1024 positions per level)
constexpr uint32_t SMALL_SLOTS = 2048;      // shared-memory table slots (load <= 0.5)
constexpr int SMALL_MAX_LEVELS = 16;

struct SmallOut {
  uint2* nodes[SMALL_MAX_LEVELS];  // layer buffers of the levels this launch will build
};

__global__ void __launch_bounds__(1024)
small_levels_kernel(const uint32_t* __restrict__ cur_in, uint32_t n_cur, SmallOut out, uint32_t* __restrict__ counts,
                    uint32_t* __restrict__ root_out) {
  __shared__ uint32_t ptr_a[SMALL_MAX], ptr_b[SMALL_MAX / 2];
  __shared__ unsigned long long skey[SMALL_SLOTS];
  __shared__ uint32_t smin[SMALL_SLOTS];
  __shared__ uint32_t warp_cnt[32];
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint32_t i = tid; i < n_cur; i += 1024) ptr_a[i] = cur_in[i];
  uint32_t* cur = ptr_a;
  uint32_t* nxt = ptr_b;
  int level = 0;
  do {
    const uint32_t n_next = (n_cur + 1) / 2;
    for (uint32_t i = tid; i < SMALL_SLOTS; i += 1024) {
      skey[i] = EMPTY_KEY;
      smin[i] = 0xffffffffu;
    }
    __syncthreads();
    uint32_t cl = 0, cr = 0, f = 0, slot = 0;
    const bool active = tid < n_next;
    if (active) {
      const uint32_t l = cur[2 * tid];
      const uint32_t r = 2 * tid + 1 < n_cur ? cur[2 * tid + 1] : PTR_NULL;
      canonical_node(l, r, cl, cr, f);
      const unsigned long long key = ((unsigned long long)cl << 32) | cr;
      slot = hash64(key) & (SMALL_SLOTS - 1);
      for (;;) {
        const unsigned long long old = atomicCAS(&skey[slot], EMPTY_KEY, key);
        if (old == EMPTY_KEY || old == key) break;
        slot = (slot + 1) & (SMALL_SLOTS - 1);
      }
      atomicMin(&smin[slot], tid);
    }
    __syncthreads();
    const bool first = active && smin[slot] == tid;
    const uint32_t word = __ballot_sync(0xffffffffu, first);
    if (lane == 0) warp_cnt[warp] = __popc(word);
    __syncthreads();
    if (warp == 0) {
      const uint32_t v = warp_cnt[lane];
      const uint32_t x = warp_inclusive_sum(v);
      warp_cnt[lane] = x - v;
      if (lane == 31) counts[level] = x;
    }
    __syncthreads();
    if (first) {
      const uint32_t id = warp_cnt[warp] + __popc(word & ((1u << lane) - 1u));
      out.nodes[level][id] = make_uint2(cl, cr);
      nxt[tid] = finish_pointer(id, f);
    }
    __syncthreads();
    if (active && !first) nxt[tid] = finish_pointer(nxt[smin[slot]] & IDX_MASK, f);
    __syncthreads();
    // the next level reads what this one wrote
    if (cur == ptr_a) { cur = ptr_b; nxt = ptr_a; } else { cur = ptr_a; nxt = ptr_b; }
    n_cur = n_next;
    ++level;
  } while (n_cur > 1);
  if (tid == 0) *root_out = cur[0];
}

// ---- the middle of the tree in ONE cooperative launch -------------------------------------
// Levels between the small top (above) and the large bottom are launch-bound when every phase is
// its own kernel: a level of half a million positions is a few microseconds of work per phase.
// Here a grid that fits the machine walks them all; grid.sync() stands where the kernel
// boundaries were.  Tables, bitmaps and the exact singleton filter are those of the large levels.
constexpr int MID_MAX_LEVELS = 24;

struct MidLevels {
  int levels;                     // levels this launch builds
  uint2* nodes[MID_MAX_LEVELS];   // their layer buffers
};

__global__ void __launch_bounds__(LVL_THREADS)
mid_levels_kernel(uint32_t* buf_a, uint32_t* buf_b, uint32_t n_cur, MidLevels out, Slot* slots, uint32_t serial0, uint32_t* aux,
                  uint32_t* bits0, uint32_t* bits1, uint32_t* multi0, uint32_t* multi1, uint32_t parity, bool first_is_upper,
                  bool use_filter, bool locality, uint32_t* blockcnt, uint32_t chunk_off, uint32_t* counts) {
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  __shared__ uint32_t word_pref[33];
  __shared__ uint32_t red[LVL_THREADS / 32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t* chunkcnt = blockcnt + chunk_off;
  uint32_t* cur = buf_a;
  uint32_t* nxt = buf_b;
  for (int lv = 0; lv < out.levels; ++lv) {
    const uint32_t n_next = (n_cur + 1) / 2;
    const uint32_t nb = (n_next + LVL_TILE - 1) / LVL_TILE;
    const uint32_t par = (parity + lv) & 1u;
    uint32_t* first_bits = par ? bits1 : bits0;
    uint32_t* multi_bits = par ? multi1 : multi0;
    const uint32_t* child_first = par ? bits0 : bits1;
    const uint32_t* child_multi = par ? multi0 : multi1;
    // the first level of a call pairs leaf ids (or an imported array): no child bitmaps, no child count
    const bool upper = first_is_upper || lv > 0;
    const bool filter = use_filter && upper;
    LevelTable tab{slots, nullptr, nullptr, (uint32_t)min((unsigned long long)max(1024u, 2u * n_next), 0x1ffffffeull)};
    tab.first_bits = first_bits;
    const uint32_t* child_unique = (locality && upper) ? counts + lv - 1 : nullptr;
    // insert (the chunk totals of the previous level are no longer read: clear them for this one)
    if (lv > 0)
      for (uint32_t i = blockIdx.x * LVL_THREADS + threadIdx.x; i <= nb / CHUNK_TILES; i += gridDim.x * LVL_THREADS) chunkcnt[i] = 0u;
    for (uint32_t block = blockIdx.x; block < nb; block += gridDim.x) {
#pragma unroll 1
      for (int it = 0; it < LVL_ITERS; ++it) {
        const uint32_t p = block * LVL_TILE + it * LVL_THREADS + threadIdx.x;
        const bool skipped = p < n_next && node_insert_position(cur, n_cur, p, tab, aux, child_unique, serial0 + lv,
                                                                filter ? child_first : nullptr, child_multi);
        const uint32_t word = __ballot_sync(0xffffffffu, skipped);
        if (lane == 0 && word) atomicOr(first_bits + (p >> 5), word);
      }
    }
    grid.sync();
    // first occurrences per tile; the bitmaps of the level after this one (the child bitmaps of
    // this level, no longer needed) are cleared on the way
    for (uint32_t t = blockIdx.x * (LVL_THREADS / 32) + warp; t < nb; t += gridDim.x * (LVL_THREADS / 32))
      count_tile(first_bits, t, t, blockcnt, chunkcnt);
    {
      const uint32_t words_after = (((n_next + 1) / 2 + LVL_TILE - 1) / LVL_TILE) * (LVL_TILE / 32);
      uint32_t* za = par ? bits0 : bits1;
      uint32_t* zb = par ? multi0 : multi1;
      for (uint32_t i = blockIdx.x * LVL_THREADS + threadIdx.x; i < words_after; i += gridDim.x * LVL_THREADS) {
        za[i] = 0u;
        zb[i] = 0u;
      }
    }
    grid.sync();
    // assign
    for (uint32_t block = blockIdx.x; block < nb; block += gridDim.x) {
      __syncthreads();  // word_pref / red of the previous tile are no longer read
      const uint32_t base = tile_base(block, blockcnt, chunkcnt, red);
      uint32_t words[LVL_ITERS];
      tile_prefix(first_bits, block, n_next, words, word_pref);
      if (block == nb - 1 && threadIdx.x == 0) counts[lv] = base + word_pref[32];
      assign_tile<MODE_NODE>(block, base, words, word_pref, nxt, n_next, tab, out.nodes[lv], 0, cur, n_cur);
    }
    grid.sync();
    // resolve
    for (uint32_t block = blockIdx.x; block < nb; block += gridDim.x) {
#pragma unroll
      for (int it = 0; it < LVL_ITERS; ++it) {
        const uint32_t p = block * LVL_TILE + it * LVL_THREADS + threadIdx.x;
        if (p < n_next && !((first_bits[p >> 5] >> lane) & 1u)) {
          const uint32_t t = aux[p];
          const uint32_t q = __ldcg(&tab.slots[t & IDX_MASK].minpos);
          if (!((__ldcg(multi_bits + (q >> 5)) >> (q & 31u)) & 1u)) atomicOr(multi_bits + (q >> 5), 1u << (q & 31));
          nxt[p] = finish_pointer(__ldcg(nxt + q) & IDX_MASK, t & ~IDX_MASK);
        }
      }
    }
    grid.sync();
    uint32_t* sw = cur;
    cur = nxt;
    nxt = sw;
    n_cur = n_next;
  }
}

// ---- host orchestration -----------------------------------------------------------

namespace {

struct LeafInput {
  const char* body = nullptr;                 // device, 16-byte aligned
  const unsigned long long* leaves = nullptr; // device
};

// Node tables: a slot's last word is an epoch tag; every node level of every build on this
// handle takes a fresh serial and sees the slots of earlier levels as empty, so the table is
// cleared only when its memory is new (or when the serials come near wrapping).
struct EpochTable {
  DevBuf<Slot> buf;
  bool cleared = false;
  uint32_t serial = 0;

  cudaError_t ensure(uint64_t slots, cudaStream_t st) {
    bool grew = false;
    const cudaError_t e = buf.ensure(slots, st, &grew);
    if (grew) cleared = false;
    return e;
  }
  int clear_if_needed(Ctx& ctx) {
    if (serial > 0xfff00000u) cleared = false;  // far from wrapping into a tag that is still in the table
    if (cleared) return STB_OK;
    Launch l(ctx, "table_clear", false);
    STB_CUDA(ctx, cudaMemsetAsync(buf.ptr, 0xff, buf.bytes(), ctx.stream));
    cleared = true;
    serial = 0;
    return STB_OK;
  }
  uint32_t take(uint32_t k) {  // the first of k fresh serials
    serial += k;
    return serial - k + 1;
  }
};

struct Scratch {
  DevBuf<uint32_t> ptr_a, ptr_b, aux, bitmask, counts, dminpos, dids;
  DevBuf<uint32_t> lvl_bits[2], lvl_multi[2];  // node levels: first occurrences / first occurrences that occur again, by level parity
  DevBuf<uint32_t> tilecnt;                    // first occurrences per tile, then per chunk of tiles (count_kernel)
  DevBuf<uint16_t> wpref;                      // rank directory of the node levels (RankDir)
  DevBuf<uint32_t> tilebase;
  DevBuf<uint32_t> leaf_done, leaf_carry;      // leaf level after a prefix: positions finished by the leaf kernel; first occurrences in the prefix
  DevBuf<Slot> side_slots;
  DevBuf<BuildFlags> flags;
  DevBuf<uint32_t> root;
  BucketWorkspace bucket;
  // profiling on: the two overflow words of every on-chip level of the current build, and each level's profile tag
  DevBuf<uint32_t> outcomes;
  std::vector<int> outcome_levels;
  // The node levels' table (the hashed leaf level uses it untagged), and the streaming build's
  // per-level tables.  They count their own epochs: a reset of one counter must never make a tag
  // that is still stored in the other table current again.
  EpochTable slots, stream_slots;

  // streaming build (host input): every chunked level keeps its own pointer array, bitmap,
  // table for the whole build, and a running total per level (two copies: a launch reads one
  // while its last tile writes the other)
  DevBuf<uint32_t> ptr_arena, bit_arena, level_sizes, run_totals;
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> chunk_events;
  DevBuf<char> stream_body;  // streaming FASTA ingest: the extracted body
  FastaStream fasta;
  int coop_grid = 0;  // CTAs of the cooperative middle launch (0 = not yet asked)
  ~Scratch() {
    for (auto e : chunk_events) cudaEventDestroy(e);
    if (copy_stream) cudaStreamDestroy(copy_stream);
  }
};

Scratch& workspace_of(Tree& t) {
  if (!t.workspace) t.workspace = std::make_shared<Scratch>();
  return *static_cast<Scratch*>(t.workspace.get());
}

// slots of the side table for leaves outside ACGT next to the direct table (side_insert)
uint32_t side_table_cap(const Tree& t, uint64_t n0) {
  return (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1024, 2 * n0), std::max<uint64_t>(1024, t.opt.side_table_slots));
}

uint32_t table_cap(uint64_t n) { return (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1024, 2 * n), 0x1ffffffeull); }
uint64_t bitmap_words(uint64_t n) { return ceil_div(n, LVL_TILE) * (LVL_TILE / 32); }

// The leaf level from ASCII text.  ACGT leaves of length 12 next to the direct table take the SWAR kernel;
// with `done_bits` (a multiple of 32 in pos0) that kernel's lookup mode.
void launch_leaf_text(Ctx& ctx, bool direct, const char* body, uint64_t n, LevelTable tab, uint32_t* tmp, BuildFlags* flags, uint32_t pos0 = 0,
                      uint32_t* done_bits = nullptr) {
  const unsigned grid = (unsigned)ceil_div(n, PACK_TILE_LEAVES);
  const size_t smem = pack_smem_bytes(ctx.S);
  Launch l(ctx, "leaf_insert");
  if (ctx.S == 12 && direct && done_bits)
    leaf_insert_acgt12_kernel<true><<<grid, PACK_THREADS, smem, ctx.stream>>>(body, n, tab, tmp, flags, pos0, done_bits);
  else if (ctx.S == 12 && direct) leaf_insert_acgt12_kernel<false><<<grid, PACK_THREADS, smem, ctx.stream>>>(body, n, tab, tmp, flags, pos0, nullptr);
  else if (ctx.S == 12) leaf_insert_text_kernel<12, false><<<grid, PACK_THREADS, smem, ctx.stream>>>(body, n, ctx.S, tab, tmp, flags, pos0);
  else if (direct) leaf_insert_text_kernel<0, true><<<grid, PACK_THREADS, smem, ctx.stream>>>(body, n, ctx.S, tab, tmp, flags, pos0);
  else leaf_insert_text_kernel<0, false><<<grid, PACK_THREADS, smem, ctx.stream>>>(body, n, ctx.S, tab, tmp, flags, pos0);
}

const BuildFlags NO_FLAGS{~0ull, 0u, 0u, 0u, 0u};

int reset_flags(Ctx& ctx, BuildFlags* flags) {
  STB_CUDA(ctx, cudaMemcpyAsync(flags, &NO_FLAGS, sizeof(NO_FLAGS), cudaMemcpyHostToDevice, ctx.stream));
  return STB_OK;
}

// The input errors the leaf kernels report (non_acgt is not one: the caller decides what it means).
int check_flags(const Ctx& ctx, const BuildFlags& flags) {
  if (flags.bad_symbol != ~0ull) return ctx.fail(STB_ERR_UNKNOWN_SYMBOL, unknown_symbol_message((int)(flags.bad_symbol & 0xff)));
  if (flags.bad_leaf) return ctx.fail(STB_ERR_BAD_LEAF, "packed leaf has bits set at or above 4*dna_size");
  return STB_OK;
}

// Tiles [first, first + count) of a level.  `carry` (null: 0) is the level's number of first
// occurrences before them, `total` receives the number up to their end.
struct TileWindow {
  uint32_t first, count;
  const uint32_t* carry;
  uint32_t* total;
};
TileWindow whole_level(uint64_t n, uint32_t* total) { return {0u, (uint32_t)ceil_div(n, LVL_TILE), nullptr, total}; }

// count -> assign -> resolve over a window of one level whose inserts are already queued.  `aux` is
// what the inserts left per position, `out` receives the finished pointers (the same array for the
// leaf level); assign and resolve see positions below n_assign and n_resolve.
// `dir` (node levels, a whole level, aux != out, n_assign == n_resolve): count (with the word
// prefixes) -> tile bases -> assign_resolve instead.
template <int MODE>
int finish_level(Ctx& ctx, const TileWindow& w, const uint32_t* aux, uint32_t* out, uint32_t n_assign, uint32_t n_resolve, LevelTable tab,
                 const uint32_t* bitmask, uint32_t* tilecnt, void* uniq, const uint32_t* children = nullptr, uint32_t n_children = 0,
                 uint32_t* multi_bits = nullptr, const uint32_t* firstpos_unless = nullptr, bool skip_resolve = false, const RankDir* dir = nullptr) {
  uint32_t* chunkcnt = tilecnt + w.count;
  STB_CUDA(ctx, cudaMemsetAsync(chunkcnt, 0, (w.count / CHUNK_TILES + 1) * 4, ctx.stream));
  {
    Launch l(ctx, "count_firsts");
    count_kernel<<<(unsigned)ceil_div((uint64_t)w.count * 32, 256), 256, 0, ctx.stream>>>(bitmask, w.first, w.count, tilecnt, chunkcnt,
                                                                                          dir ? dir->wpref : nullptr);
  }
  if (MODE == MODE_NODE && dir) {
    {
      Launch l(ctx, "tile_bases");
      tile_bases_kernel<<<(unsigned)ceil_div(w.count, CHUNK_TILES), CHUNK_TILES, 0, ctx.stream>>>(tilecnt, chunkcnt, w.count, dir->tilebase, w.total);
    }
    Launch l(ctx, "assign_resolve");
    assign_resolve_kernel<<<w.count, LVL_THREADS, 0, ctx.stream>>>(aux, out, n_assign, tab, bitmask, *dir, multi_bits, firstpos_unless, uniq, children,
                                                                    n_children);
    return STB_OK;
  }
  {
    Launch l(ctx, "assign_ids");
    assign_kernel<MODE><<<w.count, LVL_THREADS, 0, ctx.stream>>>(out, n_assign, tab, bitmask, tilecnt, chunkcnt, w.first, w.carry, w.total, uniq, ctx.S,
                                                                 children, n_children);
  }
  if (!skip_resolve) {
    Launch l(ctx, "resolve_ids");
    if (MODE == MODE_LEAF_DIRECT)
      resolve_kernel<RESOLVE_DIRECT><<<w.count, LVL_THREADS, 0, ctx.stream>>>(aux, out, n_resolve, tab, bitmask, w.first, multi_bits, firstpos_unless);
    else resolve_kernel<RESOLVE_TABLE><<<w.count, LVL_THREADS, 0, ctx.stream>>>(aux, out, n_resolve, tab, bitmask, w.first, multi_bits, firstpos_unless);
  }
  return STB_OK;
}

// Everything run_node_levels needs for a pointer array of n_cur entries.
int reserve_node_workspace(Tree& t, Scratch& sc, uint64_t n_cur) {
  cudaStream_t st = t.stream;
  const uint64_t n1 = ceil_div(n_cur, 2), n2 = ceil_div(n1, 2);
  STB_CUDA(t, sc.ptr_a.ensure(n_cur, st));
  STB_CUDA(t, sc.ptr_b.ensure(n1, st));
  STB_CUDA(t, sc.aux.ensure(n1, st));
  STB_CUDA(t, sc.lvl_bits[0].ensure(bitmap_words(n1), st));
  STB_CUDA(t, sc.lvl_multi[0].ensure(bitmap_words(n1), st));
  STB_CUDA(t, sc.lvl_bits[1].ensure(bitmap_words(n2), st));
  STB_CUDA(t, sc.lvl_multi[1].ensure(bitmap_words(n2), st));
  {
    const uint64_t tiles = ceil_div(n_cur, LVL_TILE);
    STB_CUDA(t, sc.tilecnt.ensure(tiles + tiles / CHUNK_TILES + 2, st));
  }
  STB_CUDA(t, sc.wpref.ensure(bitmap_words(n1), st));
  STB_CUDA(t, sc.tilebase.ensure(ceil_div(n1, LVL_TILE), st));
  STB_CUDA(t, sc.counts.ensure(80, st));
  STB_CUDA(t, sc.root.ensure(1, st));
  STB_CUDA(t, sc.slots.ensure((uint64_t)table_cap(n1) + 1, st));
  if (n1 >= t.opt.bucket_min && t.opt.bucket_levels > 0) {
    const BucketPlan pl = bucket_plan(n1, t.opt);  // the largest level: later ones fit in what it reserves
    if (pl.usable) STB_TRY(bucket_reserve(t, sc.bucket, pl));
  }
  return STB_OK;
}

// On-chip levels whose outcome one build can report (a build has fewer than 32 node levels).
constexpr size_t MAX_OUTCOMES = 64;

// The profile class of an on-chip level's outcome, from its two overflow words (bucket.cu: exact_pass_wanted).
const char* dedup_outcome(uint32_t first, uint32_t exact) {
  if (first == 1u) return "dedup_fallback_first_pass";
  if (first != 0u) return "dedup_fallback_distinct";
  if (exact == 2u) return "dedup_chunked";
  return exact ? "dedup_exact" : "dedup_on_chip";
}

// The on-chip (bucketed) plan of node level `level` with n_next positions, or an unusable one.
BucketPlan level_bucket_plan(const Tree& t, uint64_t n_next, int level) {
  return (n_next >= t.opt.bucket_min && (uint64_t)level < t.opt.bucket_levels) ? bucket_plan(n_next, t.opt) : BucketPlan{};
}

// Node levels from a pointer array down to a single root pointer.  Appends one layer per
// level to t.layers; counts_dev[level] receives each layer's size; returns the buffer that
// holds the root pointer in *root_buf.  The workspace must have been reserved for n_cur.
// `leaf` (optional): `cur` holds leaf words whose later occurrences are still unresolved; the first level is then
// bucketed (the caller checked level_bucket_plan) and its partition pass finishes them (LeafFinish).
int run_node_levels(Tree& t, Scratch& sc, uint32_t* cur, uint32_t* nxt, uint64_t n_cur, uint32_t* counts_dev, uint32_t** root_buf,
                    const LeafFinish* leaf = nullptr) {
  cudaStream_t st = t.stream;
  int level = 0;
  STB_TRY(sc.slots.clear_if_needed(t));  // never cleared between levels (EpochTable)
  sc.outcome_levels.clear();
  const int level_tag0 = t.profile_level;  // the caller's level of `cur` (leaf pointers: 0), or -1
  do {
    if (level_tag0 >= 0) t.profile_level = level_tag0 + level + 1;
    if (n_cur <= SMALL_MAX) {  // the rest of the tree in one launch
      SmallOut out{};
      int extra = 0;
      for (uint64_t n = n_cur;;) {
        n = ceil_div(n, 2);
        t.layers.emplace_back();
        STB_CUDA(t, t.layers.back().nodes.alloc(n, st));
        out.nodes[extra++] = t.layers.back().nodes.ptr;
        if (n <= 1) break;
      }
      Launch l(t, "small_levels");
      small_levels_kernel<<<1, 1024, 0, st>>>(cur, (uint32_t)n_cur, out, counts_dev + level, sc.root.ptr);
      level += extra;
      cur = sc.root.ptr;
      break;
    }
    const uint32_t par = (uint32_t)level & 1u;
    const uint64_t n_next = ceil_div(n_cur, 2);
    const BucketPlan pl = level_bucket_plan(t, n_next, level);
    if (!pl.usable && n_cur <= t.opt.coop_max) {  // the middle of the tree in one cooperative launch
      if (sc.coop_grid == 0) {
        int per_sm = 0, sms = 0;
        STB_CUDA(t, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mid_levels_kernel, LVL_THREADS, 0));
        STB_CUDA(t, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, t.device));
        sc.coop_grid = std::max(1, std::min(per_sm, 4) * sms);
      }
      MidLevels out{};
      uint64_t n = n_cur;
      while (n > SMALL_MAX && out.levels < MID_MAX_LEVELS) {
        n = ceil_div(n, 2);
        t.layers.emplace_back();
        STB_CUDA(t, t.layers.back().nodes.alloc(n, st));
        out.nodes[out.levels++] = t.layers.back().nodes.ptr;
      }
      const uint64_t n_first = ceil_div(n_cur, 2);
      STB_CUDA(t, cudaMemsetAsync(sc.lvl_bits[par].ptr, 0, bitmap_words(n_first) * 4, st));
      STB_CUDA(t, cudaMemsetAsync(sc.lvl_multi[par].ptr, 0, bitmap_words(n_first) * 4, st));
      uint32_t n_cur32 = (uint32_t)n_cur, serial0 = sc.slots.take((uint32_t)out.levels), parity = par;
      bool first_is_upper = level > 0, use_filter = t.opt.child_filter != 0, locality = t.opt.locality != 0;
      Slot* slots = sc.slots.buf.ptr;
      uint32_t *aux = sc.aux.ptr, *b0 = sc.lvl_bits[0].ptr, *b1 = sc.lvl_bits[1].ptr, *m0 = sc.lvl_multi[0].ptr, *m1 = sc.lvl_multi[1].ptr;
      uint32_t *blockcnt = sc.tilecnt.ptr, *counts = counts_dev + level;
      uint32_t chunk_off = (uint32_t)ceil_div(n_first, LVL_TILE);
      STB_CUDA(t, cudaMemsetAsync(blockcnt + chunk_off, 0, (chunk_off / CHUNK_TILES + 1) * 4, st));
      void* args[] = {&cur, &nxt, &n_cur32, &out, &slots, &serial0, &aux, &b0, &b1, &m0, &m1, &parity, &first_is_upper, &use_filter, &locality, &blockcnt,
                      &chunk_off, &counts};
      const unsigned grid = (unsigned)std::min<uint64_t>(sc.coop_grid, ceil_div(n_first, LVL_TILE));
      Launch l(t, "mid_levels");
      STB_CUDA(t, cudaLaunchCooperativeKernel((const void*)mid_levels_kernel, dim3(grid), dim3(LVL_THREADS), args, 0, st));
      if (out.levels & 1) std::swap(cur, nxt);
      n_cur = n;
      level += out.levels;
      continue;
    }
    t.layers.emplace_back();
    Layer& layer = t.layers.back();
    STB_CUDA(t, layer.nodes.alloc(n_next, st));
    uint32_t* first_bits = sc.lvl_bits[par].ptr;
    uint32_t* multi_bits = sc.lvl_multi[par].ptr;
    LevelTable nt{sc.slots.buf.ptr, nullptr, nullptr, table_cap(n_next)};
    nt.first_bits = first_bits;
    STB_CUDA(t, cudaMemsetAsync(first_bits, 0, bitmap_words(n_next) * 4, st));
    STB_CUDA(t, cudaMemsetAsync(multi_bits, 0, bitmap_words(n_next) * 4, st));
    // the exact singleton filter reads the bitmaps the level below left (not below the first level:
    // its children are leaf ids or an imported array, whose bitmaps this call has not built)
    const bool filter = level > 0 && t.opt.child_filter != 0;
    const uint32_t* child_first = filter ? sc.lvl_bits[par ^ 1u].ptr : nullptr;
    const uint32_t* child_multi = filter ? sc.lvl_multi[par ^ 1u].ptr : nullptr;
    // children of level 0 are leaf ids (or an imported array): not position-ordered
    const uint32_t* child_unique = (t.opt.locality && level > 0) ? counts_dev + level - 1 : nullptr;
    const unsigned nb = (unsigned)ceil_div(n_next, LVL_TILE);
    uint32_t* overflow = nullptr;
    if (pl.usable) {
      // on chip (bucket.cu); the hash-table kernels below then run only if a bucket overflowed
      STB_TRY(bucket_dedup_level(t, sc.bucket, pl, cur, (uint32_t)n_cur, (uint32_t)n_next, child_first, child_multi, sc.aux.ptr, first_bits, multi_bits,
                                 &overflow, level == 0 ? leaf : nullptr));
      if (t.profiling && sc.outcome_levels.size() < MAX_OUTCOMES) {  // read_back reports the outcome (dedup_outcome)
        STB_CUDA(t, sc.outcomes.ensure(2 * MAX_OUTCOMES, st));
        STB_CUDA(t, cudaMemcpyAsync(sc.outcomes.ptr + 2 * sc.outcome_levels.size(), overflow, 8, cudaMemcpyDeviceToDevice, st));
        sc.outcome_levels.push_back(t.profile_level);
      }
      Launch l(t, "bucket_fallback");
      bitmaps_reset_kernel<<<296, 256, 0, st>>>(first_bits, multi_bits, (uint32_t)bitmap_words(n_next), overflow);
    }
    {
      // Probe-then-claim measured faster than claim-first on B200 (12.0 vs 13.2 ms per 3.1 Gbp),
      // and chunking the level to keep table lines in L2 did not pay (profiles/README.md).
      Launch l(t, pl.usable ? "bucket_fallback" : "node_insert");
      node_insert_kernel<<<pl.usable ? std::min(nb, 1184u) : nb, LVL_THREADS, 0, st>>>(cur, (uint32_t)n_cur, (uint32_t)n_next, nt, sc.aux.ptr, child_unique,
                                                                                        sc.slots.take(1), child_first, child_multi, 0u, overflow);
    }
    const RankDir dir{sc.wpref.ptr, sc.tilebase.ptr};
    STB_TRY(finish_level<MODE_NODE>(t, whole_level(n_next, counts_dev + level), sc.aux.ptr, nxt, (uint32_t)n_next, (uint32_t)n_next, nt, first_bits,
                                    sc.tilecnt.ptr, layer.nodes.ptr, cur, (uint32_t)n_cur, multi_bits, overflow, false,
                                    t.opt.fused_resolve ? &dir : nullptr));
    std::swap(cur, nxt);
    n_cur = n_next;
    ++level;
  } while (n_cur > 1);
  t.profile_level = level_tag0;
  *root_buf = cur;
  return STB_OK;
}

// Copies the item counts at counts_dev (the leaves' first when `leaves`, then one per layer of
// t.layers) and the root pointer at root_dev to the host, with the build flags when `flags_dev` is
// given, and waits.  The flags are reported first, then a count at the index ceiling; the tree is
// cleared when either fails.  Otherwise fills in the counts and the root, and adds the outcome of every
// on-chip level that run_node_levels recorded (profiling on) to the profile.
int read_back(Tree& t, const uint32_t* counts_dev, bool leaves, const uint32_t* root_dev, const BuildFlags* flags_dev = nullptr) {
  cudaStream_t st = t.stream;
  Scratch& sc = workspace_of(t);
  const size_t first_layer = leaves ? 1 : 0;  // index of t.layers[0]'s count
  std::vector<uint32_t> counts(first_layer + t.layers.size());
  std::vector<uint32_t> outcomes(2 * sc.outcome_levels.size());
  BuildFlags flags = NO_FLAGS;
  uint32_t root = PTR_NULL;
  STB_CUDA(t, cudaMemcpyAsync(counts.data(), counts_dev, counts.size() * 4, cudaMemcpyDeviceToHost, st));
  if (flags_dev) STB_CUDA(t, cudaMemcpyAsync(&flags, flags_dev, sizeof(flags), cudaMemcpyDeviceToHost, st));
  STB_CUDA(t, cudaMemcpyAsync(&root, root_dev, 4, cudaMemcpyDeviceToHost, st));
  if (!outcomes.empty()) STB_CUDA(t, cudaMemcpyAsync(outcomes.data(), sc.outcomes.ptr, outcomes.size() * 4, cudaMemcpyDeviceToHost, st));
  STB_CUDA(t, cudaStreamSynchronize(st));
  STB_CUDA(t, cudaGetLastError());

  int s = check_flags(t, flags);
  if (s == STB_OK && flags.non_acgt) s = NOT_APPLICABLE;  // only the direct leaf level raises it: the input needs the hash-table one
  if (s == STB_OK)  // not for an attempt that another path repeats
    for (size_t k = 0; k < sc.outcome_levels.size(); ++k) t.account(dedup_outcome(outcomes[2 * k], outcomes[2 * k + 1]), sc.outcome_levels[k]).launches += 1;
  sc.outcome_levels.clear();
  for (uint32_t c : counts)
    if (s == STB_OK && c >= IDX_MASK) s = t.fail(STB_ERR_INDEX_CEILING, "a layer has 2^29-1 or more unique items; the pointer format cannot index it");
  if (s != STB_OK) {
    t.clear();
    return s;
  }
  if (leaves) t.n_leaves = counts[0];
  for (size_t k = 0; k < t.layers.size(); ++k) t.layers[k].count = counts[first_layer + k];
  t.root = root;
  return STB_OK;
}

// Reads back the counts, the flags and the root of a build from leaves; trims storage.
int finish_build(Tree& t, Scratch& sc, uint64_t n0, const uint32_t* cur) {
  cudaStream_t st = t.stream;
  STB_TRY(read_back(t, sc.counts.ptr, true, cur, sc.flags.ptr));
  t.width = n0;
  t.built = true;
  t.plan_valid = false;

  // Give back over-provisioned storage (worst case was one item per position).
  if (t.n_leaves * 2 < t.leaves.count) {
    DevBuf<unsigned long long> exact;
    STB_CUDA(t, exact.alloc(t.n_leaves, st));
    STB_CUDA(t, cudaMemcpyAsync(exact.ptr, t.leaves.ptr, t.n_leaves * 8, cudaMemcpyDeviceToDevice, st));
    t.leaves = std::move(exact);
  }
  for (auto& layer : t.layers) {
    if (layer.count * 2 < layer.nodes.count) {
      DevBuf<uint2> exact;
      STB_CUDA(t, exact.alloc(layer.count, st));
      STB_CUDA(t, cudaMemcpyAsync(exact.ptr, layer.nodes.ptr, layer.count * 8, cudaMemcpyDeviceToDevice, st));
      layer.nodes = std::move(exact);
    }
  }
  if (t.opt.reserve_pipeline) {  // so that the first sort_tree / decode of this handle does not stop to allocate
    STB_TRY(sort_reserve(t));
    STB_TRY(decode_reserve(t));
  }
  return STB_OK;
}

int build_impl(Tree& t, const LeafInput& in, uint64_t n0, bool direct) {
  const int S = t.S;
  cudaStream_t st = t.stream;
  Scratch& sc = workspace_of(t);
  STB_TRY(reserve_node_workspace(t, sc, n0));
  STB_CUDA(t, sc.bitmask.ensure(bitmap_words(n0), st));
  STB_CUDA(t, sc.flags.ensure(1, st));
  STB_TRY(reset_flags(t, sc.flags.ptr));

  // ---- leaf level ----
  t.profile_level = t.opt.profile_levels ? 0 : -1;
  const uint64_t direct_entries = direct ? (1ull << (2 * S)) : 0;
  const uint32_t leaf_cap = direct ? 0u : table_cap(n0);
  // the hashed leaf level uses the node table untagged: what it leaves there carries the tag
  // 0xffffffff, which is never a level's serial, so the node levels see those slots as empty
  if (!direct) STB_CUDA(t, sc.slots.ensure((uint64_t)leaf_cap + 1, st));
  LevelTable tab{sc.slots.buf.ptr, nullptr, nullptr, leaf_cap};
  tab.first_bits = sc.bitmask.ptr;
  STB_CUDA(t, cudaMemsetAsync(sc.bitmask.ptr, 0, bitmap_words(n0) * 4, st));
  if (direct) {
    STB_CUDA(t, sc.dminpos.ensure(direct_entries, st));
    STB_CUDA(t, sc.dids.ensure(direct_entries, st));
    STB_CUDA(t, sc.side_slots.ensure(side_table_cap(t, n0) + 1, st));
    tab.dminpos = sc.dminpos.ptr;
    tab.dids = sc.dids.ptr;
    tab.slots = sc.side_slots.ptr;  // leaves with symbols outside ACGT (side_insert)
    tab.cap = side_table_cap(t, n0);
    Launch l(t, "table_clear", false);
    STB_CUDA(t, cudaMemsetAsync(sc.dminpos.ptr, 0xff, direct_entries * 4, st));
    STB_CUDA(t, cudaMemsetAsync(sc.side_slots.ptr, 0xff, ((uint64_t)tab.cap + 1) * sizeof(Slot), st));
  } else {
    Launch l(t, "table_clear", false);
    STB_CUDA(t, cudaMemsetAsync(sc.slots.buf.ptr, 0xff, ((uint64_t)leaf_cap + 1) * sizeof(Slot), st));
  }
  const uint64_t leaf_store = direct ? std::min<uint64_t>(n0, direct_entries / 2 + side_table_cap(t, n0) / 2 + 2) : n0;
  STB_CUDA(t, t.leaves.alloc(leaf_store, st));

  // direct leaf level under a bucketed first node level: the later occurrences are resolved by that level's
  // partition pass (LeafFinish), not by a kernel of their own
  LeafFinish leaf_finish{sc.ptr_a.ptr, sc.bitmask.ptr, sc.dids.ptr, sc.side_slots.ptr};
  const bool fuse_leaf = direct && n0 > SMALL_MAX && level_bucket_plan(t, ceil_div(n0, 2), 0).usable;
  // ACGT text at S = 12 in two windows: the first P leaves as below, then the rest, which look up the ids the
  // prefix assigned (as in the streaming build, they are final) and finish most of their own pointers; the
  // partition pass then only finishes codes that had not occurred in the prefix.  P is whole tiles of both the
  // leaf kernel and the level kernels.
  const uint64_t prefix_log2 = std::min<uint64_t>(t.opt.leaf_prefix_log2, 40);
  const uint64_t P = 1ull << std::max<uint64_t>(prefix_log2, 10);
  const bool split = in.body && direct && S == 12 && fuse_leaf && prefix_log2 > 0 && n0 >= 2 * P;
  static_assert(1024 % LVL_TILE == 0 && 1024 % PACK_TILE_LEAVES == 0, "the smallest prefix is whole tiles");
  if (split) {
    STB_CUDA(t, sc.leaf_done.ensure(bitmap_words(n0), st));
    STB_CUDA(t, sc.leaf_carry.ensure(1, st));
    // an id that is not ~0 is final (assign_tile writes it); the suffix kernel writes every done word from P on
    STB_CUDA(t, cudaMemsetAsync(sc.dids.ptr, 0xff, direct_entries * 4, st));
    STB_CUDA(t, cudaMemsetAsync(sc.leaf_done.ptr, 0, P / 8, st));
    leaf_finish.done_bits = sc.leaf_done.ptr;
    launch_leaf_text(t, direct, in.body, P, tab, sc.ptr_a.ptr, sc.flags.ptr);
    const TileWindow prefix{0u, (uint32_t)(P / LVL_TILE), nullptr, sc.leaf_carry.ptr};
    STB_TRY(finish_level<MODE_LEAF_DIRECT>(t, prefix, sc.ptr_a.ptr, sc.ptr_a.ptr, (uint32_t)n0, (uint32_t)n0, tab, sc.bitmask.ptr, sc.tilecnt.ptr,
                                           t.leaves.ptr, nullptr, 0, nullptr, nullptr, true));
    launch_leaf_text(t, direct, in.body + P * 12, n0 - P, tab, sc.ptr_a.ptr + P, sc.flags.ptr, (uint32_t)P, sc.leaf_done.ptr);
    const TileWindow suffix{(uint32_t)(P / LVL_TILE), (uint32_t)ceil_div(n0 - P, LVL_TILE), sc.leaf_carry.ptr, sc.counts.ptr};
    STB_TRY(finish_level<MODE_LEAF_DIRECT>(t, suffix, sc.ptr_a.ptr, sc.ptr_a.ptr, (uint32_t)n0, (uint32_t)n0, tab, sc.bitmask.ptr, sc.tilecnt.ptr,
                                           t.leaves.ptr, nullptr, 0, nullptr, nullptr, true));
  } else {
    if (in.body) {
      launch_leaf_text(t, direct, in.body, n0, tab, sc.ptr_a.ptr, sc.flags.ptr);
    } else {
      Launch l(t, "leaf_insert");
      const unsigned nb = (unsigned)ceil_div(n0, LVL_THREADS);
      if (direct) leaf_insert_u64_kernel<true><<<nb, LVL_THREADS, 0, st>>>(in.leaves, (uint32_t)n0, S, tab, sc.ptr_a.ptr, sc.flags.ptr);
      else leaf_insert_u64_kernel<false><<<nb, LVL_THREADS, 0, st>>>(in.leaves, (uint32_t)n0, S, tab, sc.ptr_a.ptr, sc.flags.ptr);
    }
    const TileWindow all = whole_level(n0, sc.counts.ptr);
    if (direct)
      STB_TRY(finish_level<MODE_LEAF_DIRECT>(t, all, sc.ptr_a.ptr, sc.ptr_a.ptr, (uint32_t)n0, (uint32_t)n0, tab, sc.bitmask.ptr, sc.tilecnt.ptr,
                                             t.leaves.ptr, nullptr, 0, nullptr, nullptr, fuse_leaf));
    else
      STB_TRY(finish_level<MODE_LEAF_HASH>(t, all, sc.ptr_a.ptr, sc.ptr_a.ptr, (uint32_t)n0, (uint32_t)n0, tab, sc.bitmask.ptr, sc.tilecnt.ptr,
                                           t.leaves.ptr));
  }

  // ---- node levels ----
  t.layers.clear();
  uint32_t* cur = nullptr;
  STB_TRY(run_node_levels(t, sc, sc.ptr_a.ptr, sc.ptr_b.ptr, n0, sc.counts.ptr + 1, &cur, fuse_leaf ? &leaf_finish : nullptr));
  // `cur` now holds the single root pointer.
  t.profile_level = -1;

  return finish_build(t, sc, n0, cur);
}

// ---- streaming build from host memory --------------------------------------------------------
// Ids are first-occurrence ranks in position order, and a later position can never displace an
// earlier one, so once a chunk of positions has been inserted its first-occurrence bits and ids
// are final.  The text is therefore copied in power-of-two chunks (the reference's own streaming
// unit, include/shared_tree.h:305-316) and every chunk runs through all the levels it spans while
// the next one is still on the PCIe bus; the scan of each level simply continues from the running
// total.  Only the last chunk's work and the small top of the tree remain after the copy ends.
// (No singleton filter here: whether a child occurs again is not known before the last chunk.)
struct StreamPlan {
  int S = 12, Lc = 0;
  uint64_t C = 0;       // leaves per chunk
  uint64_t bound = 0;   // upper bound of the leaf count (allocation, table capacities, placement scaling)
  std::vector<uint64_t> n, ptr_off, bit_off, slot_off;  // per chunked level, from `bound`
  std::vector<uint32_t> serial;
};

// Allocations, clears and the per-level layout for a text of at most `bound` leaves.
int stream_begin(Tree& t, Scratch& sc, StreamPlan& sp, uint64_t bound) {
  const int S = t.S;
  cudaStream_t st = t.stream;
  sp.S = S;
  sp.bound = bound;
  const int chunk_log2 = (int)t.opt.stream_chunk_log2;
  sp.C = 1ull << chunk_log2;
  const int Lc = sp.Lc = chunk_log2 - 11;  // chunked node levels: a chunk still holds 2048 positions at the last one
  auto &n = sp.n, &ptr_off = sp.ptr_off, &bit_off = sp.bit_off, &slot_off = sp.slot_off;
  n.assign(Lc + 1, 0);
  ptr_off.assign(Lc + 2, 0);
  bit_off.assign(Lc + 2, 0);
  slot_off.assign(Lc + 2, 0);
  n[0] = bound;
  for (int j = 1; j <= Lc; ++j) n[j] = ceil_div(n[j - 1], 2);
  for (int j = 0; j <= Lc; ++j) {
    const uint64_t blocks = ceil_div(n[j], LVL_TILE);
    ptr_off[j + 1] = ptr_off[j] + blocks * LVL_TILE;
    bit_off[j + 1] = bit_off[j] + blocks * (LVL_TILE / 32);
    slot_off[j + 1] = slot_off[j] + (j == 0 ? 0 : (uint64_t)table_cap(n[j]) + 1);
  }
  const uint64_t direct_entries = 1ull << (2 * S);
  STB_CUDA(t, sc.ptr_arena.ensure(ptr_off[Lc + 1], st));
  STB_CUDA(t, sc.bit_arena.ensure(bit_off[Lc + 1], st));
  STB_CUDA(t, sc.run_totals.ensure(2 * (Lc + 1), st));
  STB_CUDA(t, sc.tilecnt.ensure(2 * ceil_div(sp.C, LVL_TILE) + 4, st));  // one chunk's tiles at a time (the node workspace below may ask for more)
  STB_CUDA(t, sc.level_sizes.ensure(Lc + 2, st));
  STB_CUDA(t, sc.flags.ensure(1, st));
  STB_CUDA(t, sc.dminpos.ensure(direct_entries, st));
  STB_CUDA(t, sc.dids.ensure(direct_entries, st));
  STB_CUDA(t, sc.side_slots.ensure(side_table_cap(t, bound) + 1, st));
  STB_CUDA(t, cudaMemsetAsync(sc.side_slots.ptr, 0xff, ((uint64_t)side_table_cap(t, bound) + 1) * sizeof(Slot), st));
  STB_TRY(reserve_node_workspace(t, sc, n[Lc]));  // the top of the tree, as in the one-shot build
  STB_CUDA(t, sc.stream_slots.ensure(slot_off[Lc + 1], st));
  STB_TRY(sc.stream_slots.clear_if_needed(t));
  STB_CUDA(t, cudaMemsetAsync(sc.bit_arena.ptr, 0, bit_off[Lc + 1] * 4, st));
  STB_CUDA(t, cudaMemsetAsync(sc.run_totals.ptr, 0, 2 * (Lc + 1) * 4, st));
  STB_CUDA(t, cudaMemsetAsync(sc.counts.ptr, 0, 80 * 4, st));
  STB_CUDA(t, cudaMemsetAsync(sc.dminpos.ptr, 0xff, direct_entries * 4, st));
  STB_TRY(reset_flags(t, sc.flags.ptr));
  {
    std::vector<uint32_t> sizes(Lc + 2, 0);
    for (int j = 0; j <= Lc; ++j) sizes[j] = (uint32_t)n[j];
    STB_CUDA(t, cudaMemcpyAsync(sc.level_sizes.ptr, sizes.data(), sizes.size() * 4, cudaMemcpyHostToDevice, st));
    STB_CUDA(t, cudaStreamSynchronize(st));  // `sizes` is stack memory
  }
  STB_CUDA(t, t.leaves.alloc(std::min<uint64_t>(bound, direct_entries / 2 + side_table_cap(t, bound) / 2 + 2), st));
  t.layers.clear();
  for (int j = 1; j <= Lc; ++j) {
    t.layers.emplace_back();
    STB_CUDA(t, t.layers.back().nodes.alloc(n[j], st));
  }
  sp.serial.assign(Lc + 1, 0);
  for (int j = 1; j <= Lc; ++j) sp.serial[j] = sc.stream_slots.take(1);
  return STB_OK;
}

// Leaves [c * C, c * C + cnt) of the body at `body` (device, the whole body's first byte) through the
// chunked levels.  `n0` is the true leaf count when this is the last chunk (the ragged right edge is
// only ever touched then), else the bound.
int stream_chunk(Tree& t, Scratch& sc, const StreamPlan& sp, const char* body, uint64_t c, uint64_t cnt, uint64_t n0) {
  const int Lc = sp.Lc;
  uint32_t* const ptrs = sc.ptr_arena.ptr;
  uint32_t* const bits = sc.bit_arena.ptr;
  LevelTable leaf_tab{sc.side_slots.ptr, sc.dminpos.ptr, sc.dids.ptr, side_table_cap(t, sp.bound)};
  leaf_tab.first_bits = bits;
  const uint64_t first = c * sp.C;
  launch_leaf_text(t, true, body + first * sp.S, cnt, leaf_tab, ptrs + first, sc.flags.ptr, (uint32_t)first);
  for (int j = 0; j <= Lc; ++j) {
    const uint64_t begin = first >> j, end = ceil_div(first + cnt, 1ull << j);
    const uint64_t n_here = ceil_div(n0, 1ull << j), n_below = j ? ceil_div(n0, 1ull << (j - 1)) : 0;
    uint32_t* lvl_ptr = ptrs + sp.ptr_off[j];
    uint32_t* lvl_bits = bits + sp.bit_off[j];
    // running total of the level: read from one copy, the new total goes to the other
    const TileWindow w{(uint32_t)(begin / LVL_TILE), (uint32_t)ceil_div(end - begin, LVL_TILE), sc.run_totals.ptr + (c & 1) * (Lc + 1) + j,
                       sc.run_totals.ptr + ((c + 1) & 1) * (Lc + 1) + j};
    if (j == 0) {
      STB_TRY(finish_level<MODE_LEAF_DIRECT>(t, w, lvl_ptr, lvl_ptr, (uint32_t)n_here, (uint32_t)std::min<uint64_t>(n_here, first + cnt), leaf_tab,
                                             lvl_bits, sc.tilecnt.ptr, t.leaves.ptr));
      continue;
    }
    LevelTable tab{sc.stream_slots.buf.ptr + sp.slot_off[j], nullptr, nullptr, table_cap(sp.n[j])};
    tab.first_bits = lvl_bits;
    {
      Launch l(t, "node_insert");
      // placement by child id above the first node layer; child ids are bounded by the child level's size
      const uint32_t* child_unique = (j > 1 && t.opt.locality) ? sc.level_sizes.ptr + (j - 1) : nullptr;
      node_insert_kernel<<<w.count, LVL_THREADS, 0, t.stream>>>(ptrs + sp.ptr_off[j - 1], (uint32_t)n_below, (uint32_t)end, tab, lvl_ptr, child_unique,
                                                                sp.serial[j], nullptr, nullptr, w.first, nullptr);
    }
    STB_TRY(finish_level<MODE_NODE>(t, w, lvl_ptr, lvl_ptr, (uint32_t)end, (uint32_t)end, tab, lvl_bits, sc.tilecnt.ptr, t.layers[j - 1].nodes.ptr,
                                    ptrs + sp.ptr_off[j - 1], (uint32_t)n_below));
  }
  return STB_OK;
}

// The top of the tree: everything above the last chunked level, as in the one-shot build.
int stream_finish(Tree& t, Scratch& sc, const StreamPlan& sp, uint64_t n0, uint64_t chunks) {
  const int Lc = sp.Lc;
  cudaStream_t st = t.stream;
  const uint64_t n_top = ceil_div(n0, 1ull << Lc);
  STB_CUDA(t, cudaMemcpyAsync(sc.counts.ptr, sc.run_totals.ptr + (chunks & 1) * (Lc + 1), (Lc + 1) * 4, cudaMemcpyDeviceToDevice, st));
  STB_CUDA(t, cudaMemcpyAsync(sc.ptr_a.ptr, sc.ptr_arena.ptr + sp.ptr_off[Lc], n_top * 4, cudaMemcpyDeviceToDevice, st));
  uint32_t* cur = nullptr;
  STB_TRY(run_node_levels(t, sc, sc.ptr_a.ptr, sc.ptr_b.ptr, n_top, sc.counts.ptr + 1 + Lc, &cur));
  return finish_build(t, sc, n0, cur);
}

// Queues the copy of host src[0, len) to dst in pieces of chunk_bytes, all at once on the copy
// stream; piece i is followed by sc.chunk_events[i], which work on the compute stream waits for.
int queue_chunk_copies(Tree& t, Scratch& sc, char* dst, const char* src, uint64_t len, uint64_t chunk_bytes) {
  const uint64_t chunks = ceil_div(len, chunk_bytes);
  if (!sc.copy_stream) STB_CUDA(t, cudaStreamCreateWithFlags(&sc.copy_stream, cudaStreamNonBlocking));
  while (sc.chunk_events.size() < chunks) {
    cudaEvent_t e;
    STB_CUDA(t, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    sc.chunk_events.push_back(e);
  }
  for (uint64_t i = 0; i < chunks; ++i) {
    const uint64_t first = i * chunk_bytes;
    STB_CUDA(t, cudaMemcpyAsync(dst + first, src + first, std::min(chunk_bytes, len - first), cudaMemcpyHostToDevice, sc.copy_stream));
    STB_CUDA(t, cudaEventRecord(sc.chunk_events[i], sc.copy_stream));
  }
  return STB_OK;
}

bool streaming_applies(const Tree& t, uint64_t n0_bound) {
  const uint64_t log2c = t.opt.stream_chunk_log2;
  if (log2c < 12 || log2c > 30 || t.S > 12) return false;
  return n0_bound >= t.opt.stream_min_chunks * (1ull << log2c) && n0_bound < (1ull << 30);
}

int build_streaming(Tree& t, const char* h_body, uint64_t body_len) {
  const int S = t.S;
  const uint64_t n0 = body_len / (uint64_t)S;
  if (!streaming_applies(t, n0)) return NOT_APPLICABLE;
  cudaStream_t st = t.stream;
  t.clear();
  Scratch& sc = workspace_of(t);
  StreamPlan sp;
  STB_CUDA(t, t.staging.ensure(n0 * (uint64_t)S + 16, st));
  STB_TRY(stream_begin(t, sc, sp, n0));
  const uint64_t C = sp.C, chunks = ceil_div(n0, C);
  char* text = t.staging.ptr;
  STB_TRY(queue_chunk_copies(t, sc, text, h_body, n0 * S, C * S));
  for (uint64_t c = 0; c < chunks; ++c) {
    STB_CUDA(t, cudaStreamWaitEvent(st, sc.chunk_events[c], 0));
    STB_TRY(stream_chunk(t, sc, sp, text, c, std::min<uint64_t>(C, n0 - c * C), n0));
  }
  return stream_finish(t, sc, sp, n0, chunks);
}

// The same for FASTA text with headers and line breaks (fasta_reader::load_buffer, src/fasta_reader.cpp:40-68,
// which overlaps reading with building through its loader thread, :92-106): the text is copied in
// chunks, every chunk is extracted as soon as it has arrived (the line automaton's state is carried
// on the device, ingest.cu), and every time the body has grown by a whole leaf chunk that chunk is built.
// The host reads one number per text chunk: how long the body has become.
int build_streaming_fasta(Tree& t, const char* h_text, uint64_t len) {
  const int S = t.S;
  const uint64_t bound = len / (uint64_t)S;
  if (!streaming_applies(t, bound)) return NOT_APPLICABLE;
  cudaStream_t st = t.stream;
  t.clear();
  Scratch& sc = workspace_of(t);
  StreamPlan sp;
  STB_CUDA(t, t.staging.ensure(len + 16, st));
  STB_CUDA(t, sc.stream_body.ensure(len + 64, st));
  STB_TRY(stream_begin(t, sc, sp, bound));
  const uint64_t C = sp.C;
  const uint64_t text_chunk = std::max<uint64_t>(FASTA_STREAM_ALIGN, (C * S / 2) & ~(FASTA_STREAM_ALIGN - 1));
  const uint64_t text_chunks = ceil_div(len, text_chunk);
  STB_TRY(fasta_stream_begin(t, sc.fasta, text_chunk));
  char* text = t.staging.ptr;
  char* body = sc.stream_body.ptr;
  STB_TRY(queue_chunk_copies(t, sc, text, h_text, len, text_chunk));
  uint64_t built = 0;  // leaf chunks already built
  uint64_t body_len = 0;
  for (uint64_t i = 0; i < text_chunks; ++i) {
    const uint64_t first = i * text_chunk, cnt = std::min<uint64_t>(text_chunk, len - first);
    STB_CUDA(t, cudaStreamWaitEvent(st, sc.chunk_events[i], 0));
    STB_TRY(fasta_stream_chunk(t, sc.fasta, text, first, cnt, body));
    STB_TRY(fasta_stream_body_len(t, sc.fasta, &body_len));
    // whole leaf chunks that are complete and are certainly not the last one
    while ((built + 1) * C * S <= body_len && (i + 1 < text_chunks || (built + 1) * C < body_len / S)) {
      STB_TRY(stream_chunk(t, sc, sp, body, built, C, bound));
      ++built;
    }
  }
  const uint64_t n0 = body_len / (uint64_t)S;
  if (n0 == 0) return t.fail(STB_ERR_EMPTY, "input holds fewer than dna_size bases");
  if (built == 0) return build_from_body(t, body, body_len);  // hardly any body: not worth (or not valid) chunking
  if (n0 > built * C) {
    STB_TRY(stream_chunk(t, sc, sp, body, built, n0 - built * C, n0));
    ++built;
  }
  return stream_finish(t, sc, sp, n0, built);
}

int build_dispatch(Tree& t, const LeafInput& in, uint64_t n0) {
  if (n0 == 0) return t.fail(STB_ERR_EMPTY, "input holds fewer than dna_size bases");
  // A node level of n positions probes a table of min(2n, 2^29-2) slots; from 2^29 positions on the
  // table could fill up (an endless probe) long before the index ceiling is reported, and a level's
  // positions share a word with three flag bits.  2^30 leaf positions = 12.9 Gbp at dna_size 12.
  if (n0 >= (1ull << 30)) return t.fail(STB_ERR_TOO_LARGE, "2^30 or more leaf positions");
  t.clear();
  const bool try_direct = t.S <= 12;
  if (try_direct) {
    const int s = build_impl(t, in, n0, true);
    if (s != NOT_APPLICABLE) return s;
  }
  if (n0 > 268000000ull)
    return t.fail(STB_ERR_TOO_LARGE, "hash-table leaf level supports at most 268M leaf positions in this version");
  return build_impl(t, in, n0, false);
}

}  // namespace

// Small top of a sharded build: node layers only, from a gathered pointer array.
int build_upper_levels(Tree& t, const uint32_t* d_ptrs, uint64_t n, bool at_least_one) {
  if (n == 0) return t.fail(STB_ERR_EMPTY, "no pointers");
  if (n > 400000000ull) return t.fail(STB_ERR_TOO_LARGE, "upper levels: too many pointers");
  t.clear();
  cudaStream_t st = t.stream;
  if (n == 1 && !at_least_one) {  // already the root
    uint32_t root = PTR_NULL;
    STB_CUDA(t, cudaMemcpyAsync(&root, d_ptrs, 4, cudaMemcpyDeviceToHost, st));
    STB_CUDA(t, cudaStreamSynchronize(st));
    t.root = root;
    t.built = true;
    return STB_OK;
  }
  Scratch& sc = workspace_of(t);
  STB_TRY(reserve_node_workspace(t, sc, n));
  STB_CUDA(t, cudaMemcpyAsync(sc.ptr_a.ptr, d_ptrs, n * 4, cudaMemcpyDeviceToDevice, st));
  uint32_t* cur = nullptr;
  STB_TRY(run_node_levels(t, sc, sc.ptr_a.ptr, sc.ptr_b.ptr, n, sc.counts.ptr, &cur));
  STB_TRY(read_back(t, sc.counts.ptr, false, cur));
  t.built = true;
  return STB_OK;
}

// ---- multi-GPU leaf level on the direct-addressed table (dist.cu drives it) ---------------
// Step 1: this rank's leaves lower the replicated table with GLOBAL positions.
int dist_leaf_direct_minpos(Ctx& ctx, const char* d_body, uint64_t n_local, uint64_t gpos0, uint32_t* dminpos, uint32_t* tmp,
                            int* non_acgt) {
  *non_acgt = 0;
  if (n_local == 0) return STB_OK;
  DevBuf<BuildFlags> flags;
  STB_CUDA(ctx, flags.alloc(1, ctx.stream));
  STB_TRY(reset_flags(ctx, flags.ptr));
  launch_leaf_text(ctx, true, d_body, n_local, LevelTable{nullptr, dminpos, nullptr, 0u}, tmp, flags.ptr, (uint32_t)gpos0);
  BuildFlags h{};
  STB_CUDA(ctx, cudaMemcpyAsync(&h, flags.ptr, sizeof(h), cudaMemcpyDeviceToHost, ctx.stream));
  STB_CUDA(ctx, cudaStreamSynchronize(ctx.stream));
  STB_CUDA(ctx, cudaGetLastError());
  STB_TRY(check_flags(ctx, h));
  *non_acgt = (int)h.non_acgt;
  return STB_OK;
}

int build_from_body(Tree& t, const char* d_body, uint64_t body_len) {
  LeafInput in;
  in.body = d_body;
  return build_dispatch(t, in, body_len / (uint64_t)t.S);
}

// Host text: overlap the copy with the build when the input is large enough; NOT_APPLICABLE (small
// input, dna_size > 12, or non-ACGT symbols): the caller copies and builds in one shot.
int build_from_host_body(Tree& t, const char* h_body, uint64_t body_len) { return build_streaming(t, h_body, body_len); }
int build_from_host_fasta(Tree& t, const char* h_text, uint64_t len) { return build_streaming_fasta(t, h_text, len); }

int build_from_leaves(Tree& t, const unsigned long long* d_leaves, uint64_t n) {
  LeafInput in;
  in.leaves = d_leaves;
  return build_dispatch(t, in, n);
}

}  // namespace stb
