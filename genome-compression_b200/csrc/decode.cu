// decode.cu — DAG expansion: sequential decode, batched random access, width.
//
// Replaces shared_tree::iterator (reference src/shared_tree.cpp:553-614), access_leaf
// (:231-236), operator[] (:268-291) and children()/width() (:252-259,
// include/shared_tree.h:165).  The reference walks one explicit DFS stack; here the
// DAG is expanded top-down one whole level per launch: the pointer array of node
// layer k becomes the pointer array of layer k-1 (a mirrored parent swaps its
// children, flags compose downwards), restricted to the positions that cover the
// requested leaf range, so decoding `count` leaves costs O(count + depth).
#include <algorithm>

#include "scan.cuh"
#include "staging.cuh"
#include "tree.h"

namespace stb {

constexpr int DEC_THREADS = 256;
constexpr int MAX_LAYERS = 40;

struct LayerPtrs {
  const uint2* nodes[MAX_LAYERS];
};

// access_leaf (src/shared_tree.cpp:231-236): stored leaf -> mirrored? -> transposed?
// mirrored = transposed(inverted) and transposed is an involution, so at most one of each is
// ever needed: (m,t) = 00 v, 01 T(v), 10 T(I(v)), 11 I(v).
__device__ __forceinline__ unsigned long long apply_leaf(unsigned long long v, uint32_t p, int S) {
  const bool m = (p & MIRROR) != 0, t = (p & TRANSPOSE) != 0;
  const unsigned long long x = m ? leaf_inverted(v, S) : v;
  return m != t ? leaf_transposed(x) : x;
}

// One expansion step.  cur[] holds the pointers of node layer `k` for positions
// [lo_cur, ...]; writes the child pointers for positions [lo_next, lo_next + n_next).
__global__ void __launch_bounds__(DEC_THREADS)
expand_kernel(const uint32_t* __restrict__ cur, unsigned long long lo_cur, const uint2* __restrict__ nodes,
              uint32_t* __restrict__ next, unsigned long long lo_next, unsigned long long n_next) {
  const unsigned long long j = (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x;
  if (j >= n_next) return;
  const unsigned long long c = lo_next + j;  // child position
  const uint32_t p = cur[(c >> 1) - lo_cur];
  uint32_t out = PTR_NULL;
  if (!ptr_is_null(p)) {
    const uint2 nd = __ldg(nodes + (p & IDX_MASK));
    const uint32_t m = (p >> 29) & 1u, t = (p >> 30) & 1u;
    const uint32_t child = (((uint32_t)c & 1u) ^ m) ? nd.y : nd.x;  // mirrored parent: right first (:606-612)
    if (!ptr_is_null(child)) out = compose(child, m, t);            // nulls are skipped before composing
  }
  next[j] = out;
}

__global__ void __launch_bounds__(DEC_THREADS)
leaves_out_kernel(const uint32_t* __restrict__ cur, unsigned long long n, const unsigned long long* __restrict__ leaves,
                  int S, unsigned long long* __restrict__ out) {
  const unsigned long long j = (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x;
  if (j >= n) return;
  const uint32_t p = cur[j];
  out[j] = ptr_is_null(p) ? 0ull : apply_leaf(__ldg(leaves + (p & IDX_MASK)), p, S);
}

// from_nac (src/dna.cpp:51-74), "SACRGBNKTWVDYHM-" indexed by the 4-bit code, four codes at a
// time: the table lives in four registers and PRMT is the lookup (a table in constant memory
// would serialise on the divergent index).  q: four codes in bits 0..15 -> their four letters.
__device__ __forceinline__ uint32_t nac_letters4(uint32_t q) {
  const uint32_t sel = q & 0x7777u;
  const uint32_t lo = __byte_perm(0x52434153u /* SACR */, 0x4b4e4247u /* GBNK */, sel);
  const uint32_t hi = __byte_perm(0x44565754u /* TWVD */, 0x2d4d4859u /* YHM- */, sel);
  return __byte_perm(lo, hi, 0x3210u + ((q & 0x8888u) >> 1));  // byte i from hi where code i has bit 3 set
}

// S letters of leaf v to (unaligned) shared memory
__device__ __forceinline__ void spell_bytes(uint8_t* o, unsigned long long v, int S) {
  for (int i = 0; i < S; i += 4) {
    const uint32_t w = nac_letters4((uint32_t)(v >> (4 * i)) & 0xffffu);
    o[i] = (uint8_t)w;
    if (i + 1 < S) o[i + 1] = (uint8_t)(w >> 8);
    if (i + 2 < S) o[i + 2] = (uint8_t)(w >> 16);
    if (i + 3 < S) o[i + 3] = (uint8_t)(w >> 24);
  }
}

constexpr int ASCII_TILE = 1024;
__global__ void __launch_bounds__(DEC_THREADS)
ascii_out_kernel(const uint32_t* __restrict__ cur, unsigned long long n, const unsigned long long* __restrict__ leaves,
                 int S, char* __restrict__ out) {
  __shared__ __align__(16) uint8_t stage[ASCII_TILE * 16 + 16];
  const unsigned long long tile_first = (unsigned long long)blockIdx.x * ASCII_TILE;
  const uint32_t here = (uint32_t)min((unsigned long long)ASCII_TILE, n - tile_first);
  const unsigned long long dst = tile_first * (unsigned long long)S;
  const uint32_t shift = (uint32_t)((reinterpret_cast<uintptr_t>(out) + dst) & 3ull);
  for (uint32_t j = threadIdx.x; j < here; j += DEC_THREADS) {
    const uint32_t p = cur[tile_first + j];
    const unsigned long long v = ptr_is_null(p) ? 0ull : apply_leaf(__ldg(leaves + (p & IDX_MASK)), p, S);
    spell_bytes(stage + shift + j * S, v, S);
  }
  __syncthreads();
  copy_out_staged<DEC_THREADS>(out + dst - shift, stage, shift, here * S);
}

// The last FUSE expansion steps and the output in one kernel: a thread takes one pointer into
// node layer FUSE-1 (2^FUSE leaves), walks its subtree in registers (1 + 2 + 4 node reads) and
// emits the leaves; the three largest intermediate pointer arrays (7/8 of the expansion's
// traffic) are never written.  Used when the tree has at least FUSE node layers.
constexpr int FUSE = 3;
constexpr int FUSE_LEAVES = 1 << FUSE;

__device__ __forceinline__ uint32_t child_of(uint2 nd, uint32_t parent, uint32_t side) {
  const uint32_t m = (parent >> 29) & 1u, t = (parent >> 30) & 1u;
  const uint32_t child = (side ^ m) ? nd.y : nd.x;  // mirrored parent: right first (:606-612)
  return ptr_is_null(child) ? PTR_NULL : compose(child, m, t);
}

// Walks the 2^FUSE-leaf subtree under p2; calls emit(slot 0..7, leaf pointer) for every present leaf.
// (Issuing all loads of a level before using any — nulls masked afterwards — was measured: slower.)
template <class Emit>
__device__ __forceinline__ void walk_subtree(uint32_t p2, const uint2* __restrict__ layer2, const uint2* __restrict__ layer1,
                                             const uint2* __restrict__ layer0, Emit emit) {
  if (ptr_is_null(p2)) return;
  const uint2 nd2 = __ldg(layer2 + (p2 & IDX_MASK));
#pragma unroll
  for (uint32_t a = 0; a < 2; ++a) {
    const uint32_t p1 = child_of(nd2, p2, a);
    if (ptr_is_null(p1)) continue;
    const uint2 nd1 = __ldg(layer1 + (p1 & IDX_MASK));
#pragma unroll
    for (uint32_t b = 0; b < 2; ++b) {
      const uint32_t p0 = child_of(nd1, p1, b);
      if (ptr_is_null(p0)) continue;
      const uint2 nd0 = __ldg(layer0 + (p0 & IDX_MASK));
#pragma unroll
      for (uint32_t c = 0; c < 2; ++c) {
        const uint32_t lp = child_of(nd0, p0, c);
        if (!ptr_is_null(lp)) emit(4 * a + 2 * b + c, lp);
      }
    }
  }
}

__global__ void __launch_bounds__(DEC_THREADS)
fused_leaves_kernel(const uint32_t* __restrict__ cur, unsigned long long lo_cur, const uint2* __restrict__ layer2,
                    const uint2* __restrict__ layer1, const uint2* __restrict__ layer0, const unsigned long long* __restrict__ leaves,
                    int S, unsigned long long first, unsigned long long count, unsigned long long* __restrict__ out) {
  const unsigned long long last = first + count - 1;
  const unsigned long long g = lo_cur + (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x;
  if (g * FUSE_LEAVES > last) return;
  walk_subtree(cur[g - lo_cur], layer2, layer1, layer0, [&](uint32_t slot, uint32_t lp) {
    const unsigned long long leaf = g * FUSE_LEAVES + slot;
    if (leaf >= first && leaf <= last) out[leaf - first] = apply_leaf(__ldg(leaves + (lp & IDX_MASK)), lp, S);
  });
}

// Packed leaves, fast path (range starting at a multiple of 8 leaves, 16-byte aligned
// destination, whole groups): 64 contiguous bytes per thread as four 16-byte stores.
__global__ void __launch_bounds__(DEC_THREADS)
fused_leaves_aligned_kernel(const uint32_t* __restrict__ cur, const uint2* __restrict__ layer2, const uint2* __restrict__ layer1,
                            const uint2* __restrict__ layer0, const unsigned long long* __restrict__ leaves, int S,
                            unsigned long long groups, ulonglong2* __restrict__ out) {
  const unsigned long long g = (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x;
  if (g >= groups) return;
  unsigned long long v[FUSE_LEAVES];
#pragma unroll
  for (int i = 0; i < FUSE_LEAVES; ++i) v[i] = 0ull;
  walk_subtree(cur[g], layer2, layer1, layer0, [&](uint32_t slot, uint32_t lp) {
    const unsigned long long x = apply_leaf(__ldg(leaves + (lp & IDX_MASK)), lp, S);
#pragma unroll
    for (int i = 0; i < FUSE_LEAVES; ++i)
      if (slot == (uint32_t)i) v[i] = x;
  });
  ulonglong2* o = out + g * (FUSE_LEAVES / 2);
#pragma unroll
  for (int q = 0; q < FUSE_LEAVES / 2; ++q) o[q] = make_ulonglong2(v[2 * q], v[2 * q + 1]);
}

// Text output, fast path (leaf size a multiple of 4, range starting at a multiple of 8 leaves,
// 16-byte aligned destination; whole groups only): the 8 leaves of a thread are 8*S contiguous
// bytes, spelled in registers and stored as 16-byte vectors.  No shared memory, so the L1 keeps
// the node lines that the four strided layer-0 loads of a warp share.
template <int S_T>
__global__ void __launch_bounds__(DEC_THREADS)
fused_ascii_aligned_kernel(const uint32_t* __restrict__ cur, const uint2* __restrict__ layer2, const uint2* __restrict__ layer1,
                           const uint2* __restrict__ layer0, const unsigned long long* __restrict__ leaves,
                           unsigned long long groups, uint4* __restrict__ out) {
  const unsigned long long g = (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x;
  if (g >= groups) return;
  unsigned long long v[FUSE_LEAVES];
#pragma unroll
  for (int i = 0; i < FUSE_LEAVES; ++i) v[i] = 0ull;
  walk_subtree(cur[g], layer2, layer1, layer0, [&](uint32_t slot, uint32_t lp) {
    const unsigned long long x = apply_leaf(__ldg(leaves + (lp & IDX_MASK)), lp, S_T);
#pragma unroll
    for (int i = 0; i < FUSE_LEAVES; ++i)
      if (slot == (uint32_t)i) v[i] = x;  // slot is a compile-time constant after unrolling
  });
  constexpr int WORDS = S_T / 4;  // words per leaf
  uint32_t w[FUSE_LEAVES * WORDS];
#pragma unroll
  for (int i = 0; i < FUSE_LEAVES; ++i)
#pragma unroll
    for (int k = 0; k < WORDS; ++k) w[i * WORDS + k] = nac_letters4((uint32_t)(v[i] >> (16 * k)) & 0xffffu);
  uint4* o = out + g * (FUSE_LEAVES * WORDS / 4);
#pragma unroll
  for (int q = 0; q < FUSE_LEAVES * WORDS / 4; ++q) o[q] = make_uint4(w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
}

// Text output in two phases so that both are free of bank conflicts: (1) thread t walks its
// subtree and parks the 8 leaf values in shared memory, transposed (slot-major); (2) the
// threads take consecutive leaves and spell them into the staged tile (word stores when the
// leaf size and the destination allow it), which leaves the SM as aligned words.
constexpr int FA_THREADS = 128;
constexpr int FA_TILE = FA_THREADS * FUSE_LEAVES;  // 1024 leaves
constexpr int FA_ROW = FA_THREADS + 2;             // slot-row stride: conflict-free reads by leaf order

__global__ void __launch_bounds__(FA_THREADS)
fused_ascii_kernel(const uint32_t* __restrict__ cur, unsigned long long lo_cur, const uint2* __restrict__ layer2,
                   const uint2* __restrict__ layer1, const uint2* __restrict__ layer0, const unsigned long long* __restrict__ leaves,
                   int S, unsigned long long first, unsigned long long count, char* __restrict__ out) {
  __shared__ unsigned long long vals[FUSE_LEAVES * FA_ROW];
  __shared__ __align__(16) uint8_t stage[FA_TILE * 16 + 16];
  const unsigned long long last = first + count - 1;
  const unsigned long long group0 = lo_cur + (unsigned long long)blockIdx.x * FA_THREADS;
  const unsigned long long tile_base = group0 * FUSE_LEAVES;
  const unsigned long long tile_lo = max(first, tile_base);
  const unsigned long long tile_hi = min(last + 1, tile_base + FA_TILE);  // > tile_lo for every launched CTA
  const unsigned long long dst = (tile_lo - first) * (unsigned long long)S;
  const uint32_t shift = (uint32_t)((reinterpret_cast<uintptr_t>(out) + dst) & 3ull);
  const unsigned long long g = group0 + threadIdx.x;
  if (g * FUSE_LEAVES <= last)
    walk_subtree(cur[g - lo_cur], layer2, layer1, layer0, [&](uint32_t slot, uint32_t lp) {
      vals[slot * FA_ROW + threadIdx.x] = apply_leaf(__ldg(leaves + (lp & IDX_MASK)), lp, S);
    });
  __syncthreads();
  const bool by_words = shift == 0 && (S & 3) == 0;
#pragma unroll
  for (int r = 0; r < FUSE_LEAVES; ++r) {
    const uint32_t l = r * FA_THREADS + threadIdx.x;  // leaf inside the tile
    const unsigned long long leaf = tile_base + l;
    if (leaf < tile_lo || leaf >= tile_hi) continue;
    const unsigned long long v = vals[(l & (FUSE_LEAVES - 1)) * FA_ROW + (l >> FUSE)];
    const uint32_t at = shift + (uint32_t)(leaf - tile_lo) * S;
    if (by_words) {
      uint32_t* o = reinterpret_cast<uint32_t*>(stage + at);
      for (int w = 0; w < S / 4; ++w) o[w] = nac_letters4((uint32_t)(v >> (16 * w)) & 0xffffu);
    } else {
      spell_bytes(stage + at, v, S);
    }
  }
  __syncthreads();
  copy_out_staged<FA_THREADS>(out + dst - shift, stage, shift, (uint32_t)(tile_hi - tile_lo) * S);
}

// operator[]'s descent (:268-291) from the root through node layers n_layers-1 .. stop: returns the pointer
// into node layer stop-1 (stop = 0: the leaf pointer) on the path to leaf `idx` (< width()).
__device__ __forceinline__ uint32_t descend(const LayerPtrs& layers, int n_layers, uint32_t root, unsigned long long idx,
                                            int stop) {
  uint32_t cur = root;
  for (int layer = n_layers - 1; layer >= stop; --layer) {
    const uint2 nd = __ldg(layers.nodes[layer] + (cur & IDX_MASK));
    const uint32_t m = (cur >> 29) & 1u, t = (cur >> 30) & 1u;
    const unsigned long long size = 1ull << layer;  // leaves under the logical left child (:272)
    uint32_t side = 0;
    if (idx >= size) {
      idx -= size;
      side = 1;
    }
    const uint32_t child = (side ^ m) ? nd.y : nd.x;
    cur = compose(child, m, t);
  }
  return cur;
}

// operator[] batched: one thread per query, depth dependent gathers.
__global__ void __launch_bounds__(DEC_THREADS)
random_access_kernel(const unsigned long long* __restrict__ index, unsigned long long q, LayerPtrs layers, int n_layers,
                     uint32_t root, const unsigned long long* __restrict__ leaves, int S, unsigned long long width,
                     unsigned long long* __restrict__ out, uint32_t* __restrict__ out_of_range) {
  const unsigned long long j = (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x;
  if (j >= q) return;
  const unsigned long long idx = index[j];
  if (idx >= width) {
    *out_of_range = 1u;
    out[j] = 0ull;
    return;
  }
  const uint32_t cur = descend(layers, n_layers, root, idx, 0);
  out[j] = apply_leaf(__ldg(leaves + (cur & IDX_MASK)), cur, S);
}

// ---- region extraction ------------------------------------------------------------------------
// A work item is one (region, aligned group of FUSE_LEAVES leaves the region touches).  A region's items are
// numbered in output order: first group to last on strand 0, last group to first on strand 1, so the items
// [t0, t1) of a CTA write one contiguous byte range.  Scratch per region: item base and output offset
// (exclusive scans of the item counts and of the lengths; RC_THREADS-region blocks first, then the block
// totals, then the sum of the two).
constexpr int RC_THREADS = 1024;
constexpr int RX_THREADS = 128;
// bits of the flag word the count kernel raises
constexpr unsigned long long REGION_BAD_ORDER = 1, REGION_BAD_END = 2, REGION_BAD_STRAND = 4;
// Regions of at least this many bases take their groups' pointers from one level expansion (expand_levels) over
// the hull of all such regions of the call instead of descending from the root per group.  One expansion costs a
// fixed chain of about 25 launches, which only regions this long repay; on the config-3 tree it takes the
// whole sequence as 24 regions from 4.66 to 4.60 ms (DESIGN.md, profiles/r05_regions_3100mbp*.json).
constexpr unsigned long long REGION_EXPAND_MIN = 1ull << 25;

__global__ void __launch_bounds__(RC_THREADS)
region_count_kernel(const unsigned long long* __restrict__ start, const unsigned long long* __restrict__ end,
                    const uint8_t* __restrict__ strand, unsigned long long n, unsigned long long limit, int S,
                    unsigned long long long_min, unsigned long long* __restrict__ item_base,
                    unsigned long long* __restrict__ out_off, unsigned long long* __restrict__ block_items,
                    unsigned long long* __restrict__ block_len, unsigned long long* __restrict__ flags) {
  __shared__ unsigned long long warp_totals[RC_THREADS / 32];
  const unsigned long long i = (unsigned long long)blockIdx.x * RC_THREADS + threadIdx.x;
  unsigned long long len = 0, items = 0;
  if (i < n) {
    const unsigned long long s = start[i], e = end[i];
    unsigned long long bad = 0;
    if (s > e) bad |= REGION_BAD_ORDER;
    if (e > limit) bad |= REGION_BAD_END;
    if (strand && strand[i] > 1) bad |= REGION_BAD_STRAND;
    if (bad) {
      atomicOr(flags, bad);
    } else if (e > s) {
      len = e - s;
      const unsigned long long g0 = (s / (unsigned)S) >> FUSE, g1 = ((e - 1) / (unsigned)S) >> FUSE;
      items = g1 - g0 + 1;
      if (len >= long_min) {  // flags[1] = last group of the hull, flags[2] = ~its first group (0: no hull)
        atomicMax(flags + 1, g1);
        atomicMax(flags + 2, ~g0);
      }
    }
  }
  unsigned long long total;
  const unsigned long long ib = block_exclusive_sum<RC_THREADS>(items, warp_totals, &total);
  if (i < n) item_base[i] = ib;
  if (threadIdx.x == 0) block_items[blockIdx.x] = total;
  __syncthreads();  // warp_totals is written again
  const unsigned long long ob = block_exclusive_sum<RC_THREADS>(len, warp_totals, &total);
  if (i < n) out_off[i] = ob;
  if (threadIdx.x == 0) block_len[blockIdx.x] = total;
}

// One CTA: the block totals become block bases; summary[0] = total length, summary[1] = total items.
__global__ void __launch_bounds__(1024)
region_scan_kernel(unsigned long long* __restrict__ block_items, unsigned long long* __restrict__ block_len, uint32_t blocks,
                   unsigned long long* __restrict__ summary) {
  const unsigned long long items = cta_exclusive_scan(block_items, block_items, blocks);
  const unsigned long long len = cta_exclusive_scan(block_len, block_len, blocks);
  if (threadIdx.x == 0) {
    summary[0] = len;
    summary[1] = items;
  }
}

__global__ void __launch_bounds__(RC_THREADS)
region_base_kernel(unsigned long long* __restrict__ item_base, unsigned long long* __restrict__ out_off,
                   const unsigned long long* __restrict__ block_items, const unsigned long long* __restrict__ block_len,
                   unsigned long long n) {
  const unsigned long long i = (unsigned long long)blockIdx.x * RC_THREADS + threadIdx.x;
  if (i >= n) return;
  item_base[i] += block_items[blockIdx.x];
  out_off[i] += block_len[blockIdx.x];
}

// Thread = item: finds its region (the last one whose item base is <= the item), takes the group's pointer
// into node layer FUSE-1 from the hull's expansion (regions of at least long_min bases) or on operator[]'s path
// (or, in trees of fewer than FUSE node layers, each leaf's pointer),
// walks the group, and spells the bases inside the region into the CTA's staged range, strand 1 through
// leaf_inverted and in reverse order.  The range leaves the SM as aligned words.
__global__ void __launch_bounds__(RX_THREADS)
extract_regions_kernel(const unsigned long long* __restrict__ start, const unsigned long long* __restrict__ end,
                       const uint8_t* __restrict__ strand, const unsigned long long* __restrict__ item_base,
                       const unsigned long long* __restrict__ out_off, unsigned long long n_regions, unsigned long long n_items,
                       LayerPtrs layers, int n_layers, uint32_t root, const unsigned long long* __restrict__ leaves, int S,
                       unsigned long long width, const uint32_t* __restrict__ hull, unsigned long long hull_lo,
                       unsigned long long long_min, char* __restrict__ out) {
  __shared__ __align__(16) uint8_t stage[RX_THREADS * FUSE_LEAVES * 16 + 16];
  __shared__ unsigned long long range[2];  // the CTA's output bytes [range[0], range[1])
  const unsigned long long item = (unsigned long long)blockIdx.x * RX_THREADS + threadIdx.x;
  const bool active = item < n_items;
  unsigned long long lo = 0, hi = 0, o_start = 0, g = 0;
  bool rev = false;
  unsigned long long v[FUSE_LEAVES];
#pragma unroll
  for (int i = 0; i < FUSE_LEAVES; ++i) v[i] = 0ull;
  if (active) {
    unsigned long long a = 0, b = n_regions;  // item_base[a] <= item < item_base[b] (item_base[n_regions] = n_items)
    while (b - a > 1) {
      const unsigned long long mid = a + (b - a) / 2;
      if (item_base[mid] <= item) a = mid;
      else b = mid;
    }
    const unsigned long long s = start[a], e = end[a];
    rev = strand && strand[a];
    const unsigned long long span = (unsigned long long)S * FUSE_LEAVES;  // bases of a group
    const unsigned long long j = item - item_base[a];
    g = rev ? ((e - 1) / (unsigned)S >> FUSE) - j : (s / (unsigned)S >> FUSE) + j;
    lo = max(s, g * span);
    hi = min(e, g * span + span);
    o_start = out_off[a] + (rev ? e - hi : lo - s);
    if (threadIdx.x == 0) range[0] = o_start;
    if (item + 1 == n_items || threadIdx.x == RX_THREADS - 1) range[1] = o_start + (hi - lo);
    const unsigned long long first_leaf = g * FUSE_LEAVES;
    auto wanted = [&](uint32_t slot) {  // does leaf `slot` of the group hold a base of [lo, hi)?
      const unsigned long long b0 = (first_leaf + slot) * (unsigned)S;
      return b0 < hi && b0 + (unsigned)S > lo;
    };
    if (n_layers >= FUSE) {
      const uint32_t p2 = e - s >= long_min ? hull[g - hull_lo] : descend(layers, n_layers, root, first_leaf, FUSE);
      walk_subtree(p2, layers.nodes[2], layers.nodes[1], layers.nodes[0],
                   [&](uint32_t slot, uint32_t lp) {
                     if (!wanted(slot)) return;
                     const unsigned long long x = apply_leaf(__ldg(leaves + (lp & IDX_MASK)), lp, S);
#pragma unroll
                     for (int i = 0; i < FUSE_LEAVES; ++i)
                       if (slot == (uint32_t)i) v[i] = x;
                   });
    } else {  // at most 2^n_layers < FUSE_LEAVES leaves, all in group 0
#pragma unroll
      for (int i = 0; i < FUSE_LEAVES; ++i)
        if (i < width && wanted(i)) {
          const uint32_t lp = descend(layers, n_layers, root, i, 0);
          v[i] = apply_leaf(__ldg(leaves + (lp & IDX_MASK)), lp, S);
        }
    }
  }
  __syncthreads();
  const unsigned long long base = range[0];
  const uint32_t shift = (uint32_t)((reinterpret_cast<uintptr_t>(out) + base) & 3ull);
  if (active) {
#pragma unroll
    for (int i = 0; i < FUSE_LEAVES; ++i) {
      const unsigned long long b0 = (g * FUSE_LEAVES + i) * (unsigned)S;  // first base of the leaf
      const unsigned long long a = max(lo, b0), b = min(hi, b0 + (unsigned)S);
      if (a >= b) continue;
      if (rev) {  // leaf_inverted's letter k is the complement of base b0 + S-1-k
        const uint32_t at = shift + (uint32_t)(o_start + (hi - b) - base);
        spell_bytes(stage + at, leaf_inverted(v[i], S) >> (4 * (b0 + S - b)), (int)(b - a));
      } else {
        const uint32_t at = shift + (uint32_t)(o_start + (a - lo) - base);
        spell_bytes(stage + at, v[i] >> (4 * (a - b0)), (int)(b - a));
      }
    }
  }
  __syncthreads();
  copy_out_staged<RX_THREADS>(out + base - shift, stage, shift, (uint32_t)(range[1] - base));
}

// width() for a tree that was not built here: nulls exist only on the logical right
// edge, so walk that edge: a present second child means the first subtree is full.
// A node whose children are both null is never followed: *out = WIDTH_NULL_WALK instead.
constexpr unsigned long long WIDTH_NULL_WALK = ~0ull;
__global__ void width_kernel(LayerPtrs layers, int n_layers, uint32_t root, unsigned long long* __restrict__ out) {
  if (threadIdx.x || blockIdx.x) return;
  unsigned long long w = 0;
  uint32_t cur = root;
  if (ptr_is_null(cur)) {
    *out = 0;
    return;
  }
  for (int layer = n_layers - 1; layer >= 0; --layer) {
    const uint2 nd = layers.nodes[layer][cur & IDX_MASK];
    const uint32_t m = (cur >> 29) & 1u, t = (cur >> 30) & 1u;
    const uint32_t first = m ? nd.y : nd.x, second = m ? nd.x : nd.y;
    if (!ptr_is_null(second)) {
      w += 1ull << layer;
      cur = compose(second, m, t);
    } else {
      // tested before composing: under a mirrored parent compose() sets the mirror bit of a null
      // (a stream's null carries no invariant bit), and ptr_is_null would no longer see it
      if (ptr_is_null(first)) {
        *out = WIDTH_NULL_WALK;
        return;
      }
      cur = compose(first, m, t);
    }
  }
  *out = w + 1;
}

// ---- host --------------------------------------------------------------------------

static int layer_ptrs(const Tree& t, LayerPtrs& lp) {
  if (t.layers.size() > MAX_LAYERS) return t.fail(STB_ERR_INVALID_ARG, "too many layers");
  for (size_t k = 0; k < t.layers.size(); ++k) lp.nodes[k] = t.layers[k].nodes.ptr;
  return STB_OK;
}

int compute_width(Tree& t) {
  LayerPtrs lp{};
  STB_TRY(layer_ptrs(t, lp));
  DevBuf<unsigned long long> d;
  STB_CUDA(t, d.alloc(1, t.stream));
  {
    Launch l(t, "width_walk");
    width_kernel<<<1, 32, 0, t.stream>>>(lp, (int)t.layers.size(), t.root, d.ptr);
  }
  unsigned long long w = 0;
  STB_CUDA(t, cudaMemcpyAsync(&w, d.ptr, 8, cudaMemcpyDeviceToHost, t.stream));
  STB_CUDA(t, cudaStreamSynchronize(t.stream));
  STB_CUDA(t, cudaGetLastError());
  if (w == WIDTH_NULL_WALK) return t.fail(STB_ERR_BAD_STREAM, "a node on the right edge has no child: both are null");
  t.width = w;
  return STB_OK;
}

int decode_reserve(Tree& t) {
  if (!t.built || t.width == 0) return STB_OK;
  const int stop = (int)t.layers.size() >= FUSE ? FUSE : 0;
  const uint64_t widest = (((t.width - 1) >> stop) + 1) * (stop ? 1 : 2) + 2;
  STB_CUDA(t, t.decode_a.ensure(widest, t.stream));
  STB_CUDA(t, t.decode_b.ensure(widest, t.stream));
  return STB_OK;
}

// The top-down expansion over leaves [first, last] down to pointer level stop-1 (pointer level k refers to node
// layer k and covers 2^(k+1) leaves; level -1 = leaf pointers): *cur receives that level's array (t.decode_a or
// t.decode_b), whose entry 0 is position *lo_cur.  Enqueued only: the caller synchronises before t.root may change.
static int expand_levels(Tree& t, uint64_t first, uint64_t last, int stop, uint32_t** cur_out, uint64_t* lo_out) {
  cudaStream_t st = t.stream;
  const int L = (int)t.layers.size();
  // the largest pointer array that is ever materialised: the last one
  const uint64_t widest = ((last >> stop) - (first >> stop) + 1) * (stop ? 1 : 2) + 2;
  STB_CUDA(t, t.decode_a.ensure(widest, st));
  STB_CUDA(t, t.decode_b.ensure(widest, st));
  uint32_t* cur = t.decode_a.ptr;
  uint32_t* nxt = t.decode_b.ptr;
  STB_CUDA(t, cudaMemcpyAsync(cur, &t.root, 4, cudaMemcpyHostToDevice, st));
  uint64_t lo_cur = 0;
  for (int k = L - 1; k >= stop; --k) {
    const uint64_t lo_next = first >> k, hi_next = last >> k;
    const uint64_t n_next = hi_next - lo_next + 1;
    {
      Launch l(t, "expand_level");
      expand_kernel<<<(unsigned)ceil_div(n_next, DEC_THREADS), DEC_THREADS, 0, st>>>(cur, lo_cur, t.layers[k].nodes.ptr, nxt, lo_next, n_next);
    }
    std::swap(cur, nxt);
    lo_cur = lo_next;
  }
  *cur_out = cur;
  *lo_out = lo_cur;
  return STB_OK;
}

int decode_range(const Tree& tc, uint64_t first, uint64_t count, unsigned long long* d_out, char* d_ascii) {
  Tree& t = const_cast<Tree&>(tc);
  if (!t.built) return t.fail(STB_ERR_NOT_BUILT, "tree is empty");
  if (count == 0) return STB_OK;
  if (first + count > t.width || first + count < first) return t.fail(STB_ERR_OUT_OF_RANGE, "decode range exceeds width()");
  cudaStream_t st = t.stream;
  const int L = (int)t.layers.size();
  const uint64_t last = first + count - 1;
  const int stop = L >= FUSE ? FUSE : 0;  // pointer levels below `stop` are walked inside the output kernel
  uint32_t* cur = nullptr;
  uint64_t lo_cur = 0;
  STB_TRY(expand_levels(t, first, last, stop, &cur, &lo_cur));
  if (stop) {
    const uint2 *l2 = t.layers[2].nodes.ptr, *l1 = t.layers[1].nodes.ptr, *l0 = t.layers[0].nodes.ptr;
    if (d_out) {
      const bool aligned = (first & (FUSE_LEAVES - 1)) == 0 && (reinterpret_cast<uintptr_t>(d_out) & 15u) == 0;
      const uint64_t fast_groups = aligned ? count >> FUSE : 0;
      if (fast_groups) {
        Launch l(t, "leaves_out_fused_aligned");
        fused_leaves_aligned_kernel<<<(unsigned)ceil_div(fast_groups, DEC_THREADS), DEC_THREADS, 0, st>>>(
            cur, l2, l1, l0, t.leaves.ptr, t.S, fast_groups, reinterpret_cast<ulonglong2*>(d_out));
      }
      const uint64_t done = fast_groups << FUSE;
      if (done < count) {
        Launch l(t, "leaves_out_fused");
        const uint64_t rest_first = first + done, rest = count - done;
        const uint64_t rest_groups = (last >> FUSE) - (rest_first >> FUSE) + 1;
        fused_leaves_kernel<<<(unsigned)ceil_div(rest_groups, DEC_THREADS), DEC_THREADS, 0, st>>>(
            cur + ((rest_first >> FUSE) - lo_cur), rest_first >> FUSE, l2, l1, l0, t.leaves.ptr, t.S, rest_first, rest, d_out + done);
      }
    }
    if (d_ascii) {
      // whole groups through the register path when the layout allows it, the rest (or everything) staged
      uint64_t fast_groups = 0;
      const bool aligned = (first & (FUSE_LEAVES - 1)) == 0 && (reinterpret_cast<uintptr_t>(d_ascii) & 15u) == 0;
      if (aligned && (t.S == 4 || t.S == 8 || t.S == 12 || t.S == 16)) fast_groups = count >> FUSE;
      if (fast_groups) {
        Launch l(t, "ascii_out_fused_aligned");
        const unsigned nb = (unsigned)ceil_div(fast_groups, DEC_THREADS);
        uint4* o = reinterpret_cast<uint4*>(d_ascii);
        if (t.S == 4) fused_ascii_aligned_kernel<4><<<nb, DEC_THREADS, 0, st>>>(cur, l2, l1, l0, t.leaves.ptr, fast_groups, o);
        else if (t.S == 8) fused_ascii_aligned_kernel<8><<<nb, DEC_THREADS, 0, st>>>(cur, l2, l1, l0, t.leaves.ptr, fast_groups, o);
        else if (t.S == 12) fused_ascii_aligned_kernel<12><<<nb, DEC_THREADS, 0, st>>>(cur, l2, l1, l0, t.leaves.ptr, fast_groups, o);
        else fused_ascii_aligned_kernel<16><<<nb, DEC_THREADS, 0, st>>>(cur, l2, l1, l0, t.leaves.ptr, fast_groups, o);
      }
      const uint64_t done = fast_groups << FUSE;
      if (done < count) {
        Launch l(t, "ascii_out_fused");
        const uint64_t rest_first = first + done, rest = count - done;
        const uint64_t rest_groups = (last >> FUSE) - (rest_first >> FUSE) + 1;
        fused_ascii_kernel<<<(unsigned)ceil_div(rest_groups, FA_THREADS), FA_THREADS, 0, st>>>(
            cur + ((rest_first >> FUSE) - lo_cur), rest_first >> FUSE, l2, l1, l0, t.leaves.ptr, t.S, rest_first, rest,
            d_ascii + done * (uint64_t)t.S);
      }
    }
  } else {
    if (d_out) {
      Launch l(t, "leaves_out");
      leaves_out_kernel<<<(unsigned)ceil_div(count, DEC_THREADS), DEC_THREADS, 0, st>>>(cur, count, t.leaves.ptr, t.S, d_out);
    }
    if (d_ascii) {
      Launch l(t, "ascii_out");
      ascii_out_kernel<<<(unsigned)ceil_div(count, ASCII_TILE), DEC_THREADS, 0, st>>>(cur, count, t.leaves.ptr, t.S, d_ascii);
    }
  }
  STB_CUDA(t, cudaStreamSynchronize(st));  // t.root was copied from host memory above
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

int random_access(const Tree& tc, const unsigned long long* d_index, uint64_t q, unsigned long long* d_out) {
  Tree& t = const_cast<Tree&>(tc);
  if (!t.built) return t.fail(STB_ERR_NOT_BUILT, "tree is empty");
  if (q == 0) return STB_OK;
  LayerPtrs lp{};
  STB_TRY(layer_ptrs(t, lp));
  DevBuf<uint32_t> flag;
  STB_CUDA(t, flag.alloc(1, t.stream));
  STB_CUDA(t, cudaMemsetAsync(flag.ptr, 0, 4, t.stream));
  {
    Launch l(t, "random_access");
    random_access_kernel<<<(unsigned)ceil_div(q, DEC_THREADS), DEC_THREADS, 0, t.stream>>>(
        d_index, q, lp, (int)t.layers.size(), t.root, t.leaves.ptr, t.S, t.width, d_out, flag.ptr);
  }
  uint32_t h = 0;
  STB_CUDA(t, cudaMemcpyAsync(&h, flag.ptr, 4, cudaMemcpyDeviceToHost, t.stream));
  STB_CUDA(t, cudaStreamSynchronize(t.stream));
  STB_CUDA(t, cudaGetLastError());
  if (h) return t.fail(STB_ERR_OUT_OF_RANGE, "random access index >= width()");
  return STB_OK;
}

// t.region_scratch: item bases [n], output offsets [n], block bases of each [blocks], summary [5]: total length,
// total items, error flags, hull of the long regions (last group, ~first group)
static uint64_t region_blocks(uint64_t n) { return ceil_div(n, RC_THREADS); }

int region_plan(const Tree& tc, const unsigned long long* d_start, const unsigned long long* d_end, const uint8_t* d_strand,
                uint64_t n, RegionPlan* plan) {
  Tree& t = const_cast<Tree&>(tc);
  if (!t.built) return t.fail(STB_ERR_NOT_BUILT, "tree is empty");
  cudaStream_t st = t.stream;
  const uint64_t blocks = region_blocks(n);
  STB_CUDA(t, t.region_scratch.ensure(2 * n + 2 * blocks + 5, st));
  unsigned long long* item_base = t.region_scratch.ptr;
  unsigned long long* out_off = item_base + n;
  unsigned long long* block_items = out_off + n;
  unsigned long long* block_len = block_items + blocks;
  unsigned long long* summary = block_len + blocks;
  STB_CUDA(t, cudaMemsetAsync(summary + 2, 0, 3 * 8, st));
  const unsigned long long long_min = t.layers.size() >= FUSE ? REGION_EXPAND_MIN : ~0ull;
  {
    Launch l(t, "region_count");
    region_count_kernel<<<(unsigned)blocks, RC_THREADS, 0, st>>>(d_start, d_end, d_strand, n, t.width * (uint64_t)t.S, t.S,
                                                                 long_min, item_base, out_off, block_items, block_len,
                                                                 summary + 2);
  }
  {
    Launch l(t, "region_scan");
    region_scan_kernel<<<1, 1024, 0, st>>>(block_items, block_len, (uint32_t)blocks, summary);
  }
  {
    Launch l(t, "region_base");
    region_base_kernel<<<(unsigned)blocks, RC_THREADS, 0, st>>>(item_base, out_off, block_items, block_len, n);
  }
  unsigned long long h[5] = {0, 0, 0, 0, 0};
  STB_CUDA(t, cudaMemcpyAsync(h, summary, sizeof(h), cudaMemcpyDeviceToHost, st));
  STB_CUDA(t, cudaStreamSynchronize(st));
  STB_CUDA(t, cudaGetLastError());
  if (h[2] & REGION_BAD_ORDER) return t.fail(STB_ERR_INVALID_ARG, "region start > end");
  if (h[2] & REGION_BAD_STRAND) return t.fail(STB_ERR_INVALID_ARG, "region strand is neither 0 nor 1");
  if (h[2] & REGION_BAD_END) return t.fail(STB_ERR_OUT_OF_RANGE, "region end > width() * dna_size");
  plan->total_len = h[0];
  plan->items = h[1];
  plan->hull = h[4] != 0;
  plan->hull_first = ~h[4];
  plan->hull_last = h[3];
  return STB_OK;
}

int region_write(const Tree& tc, const unsigned long long* d_start, const unsigned long long* d_end, const uint8_t* d_strand,
                 uint64_t n, const RegionPlan& plan, char* d_out) {
  Tree& t = const_cast<Tree&>(tc);
  if (plan.items == 0) return STB_OK;
  LayerPtrs lp{};
  STB_TRY(layer_ptrs(t, lp));
  const unsigned long long* item_base = t.region_scratch.ptr;
  uint32_t* hull = nullptr;
  uint64_t hull_lo = 0;
  if (plan.hull)
    STB_TRY(expand_levels(t, plan.hull_first << FUSE, std::min(t.width - 1, (plan.hull_last << FUSE) + FUSE_LEAVES - 1), FUSE,
                          &hull, &hull_lo));
  {
    Launch l(t, "extract_regions");
    extract_regions_kernel<<<(unsigned)ceil_div(plan.items, RX_THREADS), RX_THREADS, 0, t.stream>>>(
        d_start, d_end, d_strand, item_base, item_base + n, n, plan.items, lp, (int)t.layers.size(), t.root, t.leaves.ptr,
        t.S, t.width, hull, hull_lo, plan.hull ? REGION_EXPAND_MIN : ~0ull, d_out);
  }
  STB_CUDA(t, cudaStreamSynchronize(t.stream));
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

}  // namespace stb
