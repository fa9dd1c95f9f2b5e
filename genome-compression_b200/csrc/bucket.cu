// bucket.cu — on-chip deduplication of one node level (tree_constructor::emplace_node,
// reference src/shared_tree.cpp:662-672, for every position of reduce_nodes, :697-712).
//
// The keys of the first node layer are pairs of leaf ids: no locality, so a hash table in HBM
// costs one random 128-byte line per touch and B200 does only 22-25 G of those per second
// (profiles/microbench).  Here the table never leaves the chip:
//
//   partition 1   every position canonicalises its node (include/shared_tree.h:115-126) and
//                 appends the record (key64, position32) to one of 2^b1 buckets chosen by the
//                 top bits of the key's hash; a CTA groups its tile by bucket in shared memory
//                 and writes whole runs                                   [HBM stream]
//   partition 2   every first-pass bucket is split again by the next b2 hash bits, so a final
//                 bucket holds ~2 K records                               [HBM stream]
//   dedup         one CTA per final bucket: records -> shared memory, open-addressing table in
//                 shared memory, min-position per key.  A record that is not its key's minimum
//                 is a later occurrence: its first-occurrence bit is cleared and aux[position] =
//                 its flags (they travel in the record's position word) | the position of the first
//                 occurrence; a first occurrence whose key
//                 occurs again is marked in the level's `multi` bitmap (the exact singleton
//                 filter of the level above reads it).                    [HBM stream + sparse REDs]
//
// Nothing depends on the order in which records reach a bucket: ids are assigned afterwards from
// the first-occurrence bitmap in position order (build.cu), exactly the reference's emplace order.
// A bucket that outgrows its region raises *overflow; the dedup kernel then does nothing and
// build.cu re-runs the level through the hash table in HBM.
#include "bucket.cuh"
#include "scan.cuh"

namespace stb {

namespace {

constexpr int PT_ITEMS = 4;                     // records per thread; a CTA tile is PT_ITEMS * its thread count
constexpr int PT_MAX_BUCKETS = 512;             // at most 9 bits per pass
static_assert(1024 * PT_ITEMS <= COLLAPSE_WINDOW, "a run's head is at most one partition tile before its positions");
constexpr size_t pt_smem(int threads) { return (size_t)threads * PT_ITEMS * (8 + 4 + 2) + 3 * PT_MAX_BUCKETS * 4; }

constexpr int DD_CAP = 3072;                    // records of a final bucket, held in registers (DD_CAP / threads each)
constexpr int DD_SLOTS = 4096;                  // shared-memory table: key 8 B + min-position 4 B per slot
constexpr size_t DD_SMEM = (size_t)DD_SLOTS * 12 + DD_SLOTS / 8;

// overflow[0]: the level cannot be deduplicated on chip - build.cu re-runs it through the table in HBM.  It is 1
// when a first-pass bucket outgrew its region and 2 when a final bucket holds more distinct keys than the
// shared-memory table.  overflow[1]: a final bucket outgrew its fixed region - the exact-size pass takes over; it
// becomes 2 once bucket_dedup_chunked_kernel has taken a bucket.  Every reader only tests for non-zero; the values
// tell the outcomes apart for the profile (build.cu: dedup_outcome).
__device__ __forceinline__ bool exact_pass_wanted(const uint32_t* overflow) { return overflow[1] != 0u && overflow[0] == 0u; }

__device__ __forceinline__ unsigned long long bucket_hash(unsigned long long key) {
  const unsigned long long h = mix64(key);
  return h ^ (h >> 29);
}

// One partition pass.  FROM_CHILDREN: the records are made here, from the child pointer array of
// the level (position p pairs cur[2p], cur[2p+1]; odd tail -> node{last, nullptr}, utility.h:17-29);
// otherwise blockIdx.y names the first-pass bucket whose records are split.
// A tile is grouped by bucket in shared memory (rank by a shared-memory atomic per record, one
// global reservation per bucket and tile) and written out one record per thread, so that the
// stores of a warp fall into a few contiguous runs.
// Sharded build: the first pass is local (positions are global: pos_base + local position; bucket d
// belongs to rank d >> bucket_shift).  PEER marks the owner's second pass, which PULLS its input: the
// segment of (bucket, source) is read from the source's memory over NVLink with the same coalesced
// loads a local segment gets (blockIdx.y = local bucket * world + source).  Nothing is pushed:
// small scattered stores over NVLink ran at a quarter of the rate of these reads.
// EXACT (the second pass again, after a final bucket outgrew its fixed region: a key with thousands of
// occurrences, e.g. the node of two all-N leaves once per N run): the first attempt has counted every final
// bucket exactly (the counter is bumped before the capacity check), so the records are scattered again into
// regions of exactly those sizes (exact_off = exclusive scan of the counts, exact_cursor = fill state).
__device__ __forceinline__ uint32_t finish_leaf(uint32_t t, const LeafFinish& leaf) {
  const uint32_t s = t & IDX_MASK;
  const uint32_t id = (s & LEAF_SIDE) ? (__ldcg(leaf.words + __ldcg(&leaf.side[s & (LEAF_SIDE - 1u)].minpos)) & IDX_MASK) : __ldcg(leaf.dids + s);
  return finish_pointer(id, t & ~IDX_MASK);
}

template <bool FROM_CHILDREN, int PT_THREADS, bool PEER, bool EXACT, bool LEAF = false>
__device__ __forceinline__ void
partition_tile(const uint32_t bx, const uint32_t by, const uint32_t* __restrict__ cur, uint32_t n_cur, uint32_t n_next,
               const unsigned long long* in_keys, const uint32_t* in_pos,
               const uint32_t* __restrict__ in_count, uint32_t in_cap,
               unsigned long long* __restrict__ out_keys, uint32_t* __restrict__ out_pos, uint32_t* __restrict__ out_count,
               uint32_t out_cap, int shift, int bits, uint32_t* __restrict__ aux, uint32_t* __restrict__ first_bits,
               uint32_t* __restrict__ multi_bits, const uint32_t* __restrict__ child_first, const uint32_t* __restrict__ child_multi,
               uint32_t* __restrict__ overflow, uint32_t segs, uint32_t pos_base, const PeerDest& peer, const uint32_t* __restrict__ exact_off,
               const LeafFinish& leaf = LeafFinish{}) {
  constexpr int PT_TILE = PT_THREADS * PT_ITEMS, PT_WARPS = PT_THREADS / 32;
  extern __shared__ __align__(16) uint8_t smem[];
  unsigned long long* skey = reinterpret_cast<unsigned long long*>(smem);
  uint32_t* spos = reinterpret_cast<uint32_t*>(smem + (size_t)PT_TILE * 8);
  uint32_t* hist = spos + PT_TILE;
  uint32_t* loff = hist + PT_MAX_BUCKETS;
  uint32_t* goff = loff + PT_MAX_BUCKETS;
  uint16_t* sdig = reinterpret_cast<uint16_t*>(goff + PT_MAX_BUCKETS);
  __shared__ uint32_t warp_totals[PT_WARPS];

  const uint32_t tid = threadIdx.x, lane = tid & 31;
  const uint32_t nb = 1u << bits;
  uint32_t count;
  const uint32_t first = bx * PT_TILE;
  uint64_t in_base = 0;
  if (FROM_CHILDREN) {
    count = n_next;
  } else if (PEER) {
    const uint32_t src = by % peer.world, local = by / peer.world;
    const uint32_t bucket = (peer.src << peer.bucket_shift) | local;  // this owner's bucket, in the source's numbering
    count = min(peer.counts_in ? __ldg(peer.counts_in + src * peer.counts_stride + local)
                               : *reinterpret_cast<const volatile uint32_t*>(peer.base[src] + peer.count_off + 4ull * bucket), in_cap);
    if (first >= count) return;
    in_keys = reinterpret_cast<const unsigned long long*>(peer.base[src] + peer.keys_off);
    in_pos = reinterpret_cast<const uint32_t*>(peer.base[src] + peer.pos_off);
    in_base = (uint64_t)bucket * in_cap;
  } else {
    count = min(__ldg(in_count + by), in_cap);
    if (first >= count) return;
    in_base = (uint64_t)by * in_cap;
  }
  for (uint32_t i = tid; i < nb; i += PT_THREADS) hist[i] = 0;
  uint2* schild = reinterpret_cast<uint2*>(smem);  // LEAF: the tile's finished children (the staging area is not in use yet)
  if (FROM_CHILDREN && LEAF) {
    // the children are leaf words: finish the later occurrences (id from the table), write them back, and keep
    // the tile's pairs in shared memory for the neighbour comparison below
#pragma unroll
    for (int it = 0; it < PT_ITEMS; ++it) {
      const uint32_t o = it * PT_THREADS + tid, i = first + o;
      if (i < count) {
        const bool pair = 2 * (uint64_t)i + 1 < n_cur;
        uint32_t l, r = PTR_NULL;
        if (pair) {
          const uint2 pr = __ldcg(reinterpret_cast<const uint2*>(leaf.words) + i);
          l = pr.x;
          r = pr.y;
        } else {
          l = __ldcg(leaf.words + 2 * (uint64_t)i);
        }
        // (no bitmap: every word is still a code, as the sharded build's replicated leaf table leaves them)
        uint32_t finished = leaf.first_bits ? __ldg(leaf.first_bits + (i >> 4)) : 0u;
        if (leaf.done_bits) finished |= __ldg(leaf.done_bits + (i >> 4));
        finished = (finished >> ((2u * i) & 31u)) | (pair ? 0u : 2u);
        if (!(finished & 1u)) l = finish_leaf(l, leaf);
        if (!(finished & 2u)) r = finish_leaf(r, leaf);
        // only a pair with a word finished here goes back to memory
        if ((finished & 3u) != 3u) {
          if (pair) reinterpret_cast<uint2*>(leaf.words)[i] = make_uint2(l, r);
          else leaf.words[2 * (uint64_t)i] = l;
        }
        schild[o] = make_uint2(l, r);
      }
    }
  }
  __syncthreads();

  unsigned long long key[PT_ITEMS];
  uint32_t pos[PT_ITEMS], dr[PT_ITEMS];
  uint32_t flag_of[PT_ITEMS];
  bool collapsed[PT_ITEMS];
  __shared__ uint32_t shead[PT_TILE / 32];  // FROM_CHILDREN: bit per tile position, set for the positions that are not collapsed
  if (!FROM_CHILDREN) {
    // all of a thread's loads are issued before the first one is used: a segment pulled over NVLink
    // answers after a few microseconds, and only bytes in flight hide that
#pragma unroll
    for (int it = 0; it < PT_ITEMS; ++it) {
      const uint32_t i = first + it * PT_THREADS + tid;
      if (i < count) {
        key[it] = __ldcs(in_keys + in_base + i);
        pos[it] = __ldcs(in_pos + in_base + i);
      }
    }
  }
#pragma unroll
  for (int it = 0; it < PT_ITEMS; ++it) {
    const uint32_t i = first + it * PT_THREADS + tid;
    bool valid = i < count;
    dr[it] = 0xffffffffu;
    if (FROM_CHILDREN) {
      pos[it] = pos_base + i;
      uint32_t l = 0, r = 0;
      bool same = false;  // the same children as the position before it (runs of N, of one letter, of a short period)
      if (valid && LEAF) {
        const uint32_t o = it * PT_THREADS + tid;
        const uint2 pr = schild[o];
        l = pr.x;
        r = pr.y;
        if (o > 0) {
          const uint2 before = schild[o - 1];
          same = before.x == l && before.y == r;
        }
      } else if (valid) {
        if (2 * (uint64_t)i + 1 < n_cur) {
          const uint2 pr = __ldg(reinterpret_cast<const uint2*>(cur) + i);
          l = pr.x;
          r = pr.y;
        } else {
          l = cur[2 * (uint64_t)i];
          r = PTR_NULL;
        }
        if (it * PT_THREADS + tid > 0) {  // never the first position of a tile: every tile keeps a head
          const uint2 before = __ldg(reinterpret_cast<const uint2*>(cur) + i - 1);
          same = before.x == l && before.y == r;
        }
      }
      // Runs collapse here: a position that repeats its predecessor makes no record (a genome's N runs
      // would otherwise put millions of equal keys into one bucket); it is a later occurrence of the
      // run's head, which stands for the run.  Every other position starts as a first occurrence; the
      // dedup kernel clears the later ones.
      const uint32_t heads = __ballot_sync(0xffffffffu, valid && !same);
      const uint32_t word_at = (it * PT_THREADS + tid) >> 5;
      if (lane == 0) {
        shead[word_at] = heads;
        if (heads) first_bits[i >> 5] = heads;
      }
      collapsed[it] = valid && same;
      if (valid && !same && child_first) {  // a child that never repeats: the only node with that child, no record
        const uint32_t repeats = ~__ldg(child_first + (i >> 4)) | __ldg(child_multi + (i >> 4));
        valid = ((repeats >> ((2u * i) & 31u)) & 3u) == 3u;
      } else if (same) {
        valid = false;
      }
      uint32_t cl, cr, f = 0;
      if (valid || collapsed[it]) {
        canonical_node(l, r, cl, cr, f);
        key[it] = pair_key(cl, cr);
        // the flags (bits 29..31) travel in the record's position word: only a later occurrence needs them again
        // (the dedup kernel writes aux[position] = flags | first position; a first occurrence is recomputed by assign)
        if (valid) pos[it] |= f;
      }
      flag_of[it] = f;
    }
    if (valid) {
      const uint32_t d = (uint32_t)(bucket_hash(key[it]) >> shift) & (nb - 1u);
      dr[it] = (d << 16) | atomicAdd(&hist[d], 1u);
    }
  }
  __syncthreads();
  if (FROM_CHILDREN) {
#pragma unroll
    for (int it = 0; it < PT_ITEMS; ++it) {
      const uint32_t o = it * PT_THREADS + tid;  // offset in the tile
      if (collapsed[it]) {
        // the run's head: the nearest position at or before this one that is not collapsed
        uint32_t w = o >> 5;
        uint32_t m = shead[w] & (0xffffffffu >> (31u - (o & 31u)));
        while (m == 0u) m = shead[--w];
        const uint32_t head = (w << 5) + 31u - (uint32_t)__clz(m);
        aux[first + o] = flag_of[it] | (pos_base + first + head);
        if (head + 1u == o && multi_bits) atomicOr(multi_bits + ((first + head) >> 5), 1u << ((first + head) & 31u));  // the head occurs again
      }
    }
  }
  // exclusive scan of the tile's bucket counts; one global reservation per bucket
  {
    const uint32_t c = tid < nb ? hist[tid] : 0u;
    const uint32_t before = block_exclusive_sum<PT_THREADS>(c, warp_totals);
    if (tid < nb) {
      loff[tid] = before;
      uint32_t g = 0;
      if (c) {
        const uint32_t bucket = FROM_CHILDREN ? tid : (((by / segs) << bits) | tid);
        g = atomicAdd(out_count + bucket, c);  // EXACT: out_count is the fill state of the exact-size regions
        if (EXACT) g += __ldg(exact_off + bucket);
        else if (g + c > out_cap) *overflow = 1u;
      }
      goff[tid] = g;
    }
  }
  __syncthreads();
  uint32_t staged = 0;  // records of this tile (valid ones only)
#pragma unroll
  for (int it = 0; it < PT_ITEMS; ++it) {
    if (dr[it] != 0xffffffffu) {
      const uint32_t d = dr[it] >> 16, at = loff[d] + (dr[it] & 0xffffu);
      skey[at] = key[it];
      spos[at] = pos[it];
      sdig[at] = (uint16_t)d;
    }
  }
  staged = loff[nb - 1] + hist[nb - 1];
  __syncthreads();
#pragma unroll
  for (int it = 0; it < PT_ITEMS; ++it) {
    const uint32_t j = it * PT_THREADS + tid;
    if (j < staged) {
      const uint32_t d = sdig[j];
      const uint32_t at = goff[d] + (j - loff[d]);  // place in the bucket's region
      if (EXACT) {
        out_keys[at] = skey[j];
        out_pos[at] = spos[j];
      } else if (at < out_cap) {
        const uint32_t bucket = FROM_CHILDREN ? d : (((by / segs) << bits) | d);
        const uint64_t dst = (uint64_t)bucket * out_cap + at;
        out_keys[dst] = skey[j];
        out_pos[dst] = spos[j];
      }
    }
  }
}

template <bool FROM_CHILDREN, int PT_THREADS, bool PEER>
__global__ void __launch_bounds__(PT_THREADS, 2048 / PT_THREADS)
partition_kernel(const uint32_t* __restrict__ cur, uint32_t n_cur, uint32_t n_next,
                 const unsigned long long* in_keys, const uint32_t* in_pos,
                 const uint32_t* __restrict__ in_count, uint32_t in_cap,
                 unsigned long long* __restrict__ out_keys, uint32_t* __restrict__ out_pos, uint32_t* __restrict__ out_count,
                 uint32_t out_cap, int shift, int bits, uint32_t* __restrict__ aux, uint32_t* __restrict__ first_bits,
                 uint32_t* __restrict__ multi_bits, const uint32_t* __restrict__ child_first, const uint32_t* __restrict__ child_multi,
                 uint32_t* __restrict__ overflow, uint32_t segs, uint32_t pos_base, PeerDest peer) {
  partition_tile<FROM_CHILDREN, PT_THREADS, PEER, false>(blockIdx.x, blockIdx.y, cur, n_cur, n_next, in_keys, in_pos, in_count, in_cap, out_keys, out_pos,
                                                         out_count, out_cap, shift, bits, aux, first_bits, multi_bits, child_first, child_multi, overflow,
                                                         segs, pos_base, peer, nullptr);
}

// the first node level over leaf words that are finished on the way (LeafFinish)
template <int PT_THREADS>
__global__ void __launch_bounds__(PT_THREADS, 2048 / PT_THREADS)
partition_leaves_kernel(LeafFinish leaf, uint32_t n_cur, uint32_t n_next, unsigned long long* __restrict__ out_keys, uint32_t* __restrict__ out_pos,
                        uint32_t* __restrict__ out_count, uint32_t out_cap, int shift, int bits, uint32_t* __restrict__ aux, uint32_t* __restrict__ first_bits,
                        uint32_t* __restrict__ multi_bits, uint32_t* __restrict__ overflow, uint32_t pos_base) {
  partition_tile<true, PT_THREADS, false, false, true>(blockIdx.x, 0u, nullptr, n_cur, n_next, nullptr, nullptr, nullptr, 0u, out_keys, out_pos, out_count,
                                                       out_cap, shift, bits, aux, first_bits, multi_bits, nullptr, nullptr, overflow, 1u, pos_base, PeerDest{},
                                                       nullptr, leaf);
}


// exclusive scan of the final buckets' exact record counts; clears the counts (they become the fill state)
__global__ void __launch_bounds__(1024) exact_offsets_kernel(uint32_t* __restrict__ count2, uint32_t nb, uint32_t* __restrict__ off,
                                                              const uint32_t* __restrict__ overflow) {
  if (!exact_pass_wanted(overflow)) return;
  const uint32_t total = cta_exclusive_scan(count2, off, nb);
  for (uint32_t i = threadIdx.x; i < nb; i += 1024) count2[i] = 0u;  // each thread clears the counts it has read
  if (threadIdx.x == 0) off[nb] = total;
}

// the second pass again, into the exact-size regions; a grid that fits the machine walks the tiles, so the
// launch costs next to nothing when it has nothing to do
template <int PT_THREADS>
__global__ void __launch_bounds__(PT_THREADS, 2048 / PT_THREADS)
partition_exact_kernel(const unsigned long long* in_keys, const uint32_t* in_pos, const uint32_t* __restrict__ in_count, uint32_t in_cap,
                       unsigned long long* __restrict__ out_keys, uint32_t* __restrict__ out_pos, uint32_t* __restrict__ fill, int shift, int bits,
                       uint32_t* __restrict__ overflow, const uint32_t* __restrict__ exact_off, uint32_t tiles_x, uint32_t tiles_y) {
  if (!exact_pass_wanted(overflow)) return;
  for (uint32_t v = blockIdx.x; v < tiles_x * tiles_y; v += gridDim.x) {
    partition_tile<false, PT_THREADS, false, true>(v % tiles_x, v / tiles_x, nullptr, 0u, 0u, in_keys, in_pos, in_count, in_cap, out_keys, out_pos, fill, 0u,
                                                   shift, bits, nullptr, nullptr, nullptr, nullptr, nullptr, overflow, 1u, 0u, PeerDest{}, exact_off);
    __syncthreads();
  }
}

// One CTA per final bucket.  The records stay in registers; the table (key, min-position per slot)
// lives in shared memory and is never written back.
// PEER (sharded build): positions are global; position p lives on rank p >> log2_positions.  The
// answers (a later occurrence and where its key came first; a first occurrence whose key came again)
// are appended to a list per home rank in THIS rank's memory; the home ranks read their lists after
// the level's barrier and apply them to their own words (shard.cu: apply_answers_kernel).
// EXACT: the buckets lie in exact-size regions (counts = their offsets, one more than there are buckets); the
// ones that fit the registers are done here, the larger ones by bucket_dedup_chunked_kernel.
template <int DD_THREADS, bool PEER, bool EXACT = false>
__global__ void __launch_bounds__(DD_THREADS)
bucket_dedup_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ poss, const uint32_t* __restrict__ counts,
                    uint32_t cap, uint32_t* __restrict__ aux, uint32_t* __restrict__ first_bits, uint32_t* __restrict__ multi_bits,
                    const uint32_t* __restrict__ overflow, PeerHome home) {
  extern __shared__ __align__(16) uint8_t smem[];
  unsigned long long* tkey = reinterpret_cast<unsigned long long*>(smem);
  uint32_t* tmin = reinterpret_cast<uint32_t*>(smem + (size_t)DD_SLOTS * 8);  // smallest position of the slot's key
  uint32_t* tmulti = tmin + DD_SLOTS;                                         // bit per slot: the key occurred again
  constexpr int DD_ITEMS = DD_CAP / DD_THREADS;
  __shared__ uint32_t tmin_cnt[STB_MAX_RANKS], tmin_base[STB_MAX_RANKS];  // PEER: answers per home rank
  const uint32_t* overflow_out = overflow;
  if (PEER && threadIdx.x < STB_MAX_RANKS) tmin_cnt[threadIdx.x] = 0u;
  if (EXACT ? !exact_pass_wanted(overflow) : (overflow[0] || (!PEER && overflow[1]))) return;
  const uint32_t tid = threadIdx.x;
  const uint32_t count = EXACT ? __ldg(counts + blockIdx.x + 1) - __ldg(counts + blockIdx.x) : min(__ldg(counts + blockIdx.x), cap);
  if (count == 0 || (EXACT && count > (uint32_t)DD_CAP)) return;
  const uint64_t base = EXACT ? (uint64_t)__ldg(counts + blockIdx.x) : (uint64_t)blockIdx.x * cap;

  unsigned long long key[DD_ITEMS];
  uint32_t pos[DD_ITEMS];
#pragma unroll
  for (int j = 0; j < DD_ITEMS; ++j) {
    const uint32_t i = j * DD_THREADS + tid;
    if (i < count) {
      key[j] = __ldcs(keys + base + i);
      pos[j] = __ldcs(poss + base + i);
    }
  }
  // the table is as large as this bucket needs (a power of two >= 2 x its records): the level
  // above the first ones sends few records per bucket and should not pay for a full clear
  uint32_t slots = 64;
  while (slots < 2 * count && slots < DD_SLOTS) slots <<= 1;
  const uint32_t mask = slots - 1;
  for (uint32_t i = tid; i < slots; i += DD_THREADS) {
    tkey[i] = EMPTY_KEY;
    tmin[i] = 0xffffffffu;
  }
  if (tid < DD_SLOTS / 32) tmulti[tid] = 0u;
  static_assert(DD_SLOTS % DD_THREADS == 0 && DD_CAP % DD_THREADS == 0 && DD_SLOTS / 32 <= DD_THREADS, "tile shapes");
  __syncthreads();
  uint32_t slot[DD_ITEMS];
#pragma unroll
  for (int j = 0; j < DD_ITEMS; ++j) {
    const uint32_t i = j * DD_THREADS + tid;
    if (i >= count) continue;
    uint32_t h = (uint32_t)bucket_hash(key[j]) & mask;
    for (;;) {
      unsigned long long k = tkey[h];
      if (k == EMPTY_KEY) k = atomicCAS(&tkey[h], EMPTY_KEY, key[j]);
      if (k == EMPTY_KEY) break;  // claimed
      if (k == key[j]) {
        atomicOr(&tmulti[h >> 5], 1u << (h & 31));
        break;
      }
      h = (h + 1) & mask;
    }
    atomicMin(&tmin[h], pos[j] & IDX_MASK);
    slot[j] = h;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < DD_ITEMS; ++j) {
    const uint32_t i = j * DD_THREADS + tid;
    if (i >= count) continue;
    const uint32_t p = pos[j] & IDX_MASK, h = slot[j], fp = tmin[h];
    const bool later = fp != p;
    const bool again = !later && ((tmulti[h >> 5] >> (h & 31)) & 1u);
    if (PEER) {
      // answer = (flags | position) << 32 | first position, or | 0xffffffff for "this first occurrence occurs again";
      // kept in registers until the CTA has reserved room in the lists
      slot[j] = later ? fp : (again ? 0xffffffffu : 0xfffffffeu);
      if (later || again) atomicAdd(&tmin_cnt[p >> home.log2_positions], 1u);
    } else if (later) {  // a later occurrence: not a first, and it points at the first
      atomicAnd(first_bits + (p >> 5), ~(1u << (p & 31)));
      aux[p] = (pos[j] & ~IDX_MASK) | fp;
    } else if (again) {
      atomicOr(multi_bits + (p >> 5), 1u << (p & 31));
    }
  }
  if (PEER) {
    __syncthreads();
    if (tid < STB_MAX_RANKS) {  // one reservation per home rank and CTA
      const uint32_t c = tmin_cnt[tid];
      uint32_t at = 0;
      if (c) {
        at = atomicAdd(reinterpret_cast<uint32_t*>(home.base[home.self] + home.ans_count_off) + tid, c);
        if (at + c > home.ans_cap) *const_cast<uint32_t*>(overflow_out) = 1u;
      }
      tmin_base[tid] = at;
      tmin_cnt[tid] = 0u;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < DD_ITEMS; ++j) {
      const uint32_t i = j * DD_THREADS + tid;
      if (i >= count || slot[j] == 0xfffffffeu) continue;
      const uint32_t hr = (pos[j] & IDX_MASK) >> home.log2_positions;
      const uint32_t at = tmin_base[hr] + atomicAdd(&tmin_cnt[hr], 1u);
      if (at < home.ans_cap)
        reinterpret_cast<unsigned long long*>(home.base[home.self] + home.ans_off)[(uint64_t)hr * home.ans_cap + at] =
            ((unsigned long long)pos[j] << 32) | slot[j];
    }
  }
}

// The same for final buckets of any size (exact-size regions, see partition_tile): the records are walked
// twice in chunks instead of being kept in registers.  Thousands of occurrences of one key add records, not
// table entries; only a bucket with more DISTINCT keys than the table holds gives up (overflow[0]).
template <int DD_THREADS>
__global__ void __launch_bounds__(DD_THREADS)
bucket_dedup_chunked_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ poss, const uint32_t* __restrict__ off, uint32_t nb,
                            uint32_t* __restrict__ aux, uint32_t* __restrict__ first_bits, uint32_t* __restrict__ multi_bits, uint32_t* __restrict__ overflow) {
  if (!exact_pass_wanted(overflow)) return;
  extern __shared__ __align__(16) uint8_t smem[];
  unsigned long long* tkey = reinterpret_cast<unsigned long long*>(smem);
  uint32_t* tmin = reinterpret_cast<uint32_t*>(smem + (size_t)DD_SLOTS * 8);
  uint32_t* tmulti = tmin + DD_SLOTS;
  __shared__ uint32_t full;
  const uint32_t tid = threadIdx.x;
  constexpr uint32_t mask = DD_SLOTS - 1;
  for (uint32_t b = blockIdx.x; b < nb; b += gridDim.x) {
    const uint32_t base = __ldg(off + b), count = __ldg(off + b + 1) - base;
    if (count <= (uint32_t)DD_CAP) continue;  // done by bucket_dedup_kernel<.., EXACT>
    if (tid == 0) overflow[1] = 2u;
    for (uint32_t i = tid; i < DD_SLOTS; i += DD_THREADS) {
      tkey[i] = EMPTY_KEY;
      tmin[i] = 0xffffffffu;
    }
    if (tid < DD_SLOTS / 32) tmulti[tid] = 0u;
    if (tid == 0) full = 0u;
    __syncthreads();
    for (uint32_t i = tid; i < count; i += DD_THREADS) {
      const unsigned long long key = __ldg(keys + base + i);
      const uint32_t pos = __ldg(poss + base + i);
      uint32_t h = (uint32_t)bucket_hash(key) & mask, steps = 0;
      for (;;) {
        unsigned long long k = tkey[h];
        if (k == EMPTY_KEY) k = atomicCAS(&tkey[h], EMPTY_KEY, key);
        if (k == EMPTY_KEY) break;  // claimed
        if (k == key) {
          if (!((tmulti[h >> 5] >> (h & 31)) & 1u)) atomicOr(&tmulti[h >> 5], 1u << (h & 31));
          break;
        }
        h = (h + 1) & mask;
        if (++steps == DD_SLOTS) break;  // every slot holds another key
      }
      if (steps == DD_SLOTS) full = 1u;
      else if (tmin[h] > (pos & IDX_MASK)) atomicMin(&tmin[h], pos & IDX_MASK);
    }
    __syncthreads();
    if (full) {
      if (tid == 0) overflow[0] = 2u;
      return;  // the whole level is done again through the table in HBM
    }
    for (uint32_t i = tid; i < count; i += DD_THREADS) {
      const unsigned long long key = __ldg(keys + base + i);
      const uint32_t pf = __ldg(poss + base + i), p = pf & IDX_MASK;
      uint32_t h = (uint32_t)bucket_hash(key) & mask;
      while (tkey[h] != key) h = (h + 1) & mask;
      const uint32_t fp = tmin[h];
      if (fp != p) {  // a later occurrence: not a first, and it points at the first
        atomicAnd(first_bits + (p >> 5), ~(1u << (p & 31)));
        aux[p] = (pf & ~IDX_MASK) | fp;
      } else if ((tmulti[h >> 5] >> (h & 31)) & 1u) {
        atomicOr(multi_bits + (p >> 5), 1u << (p & 31));
      }
    }
    __syncthreads();
  }
}

}  // namespace

BucketPlan bucket_plan(uint64_t n, const Options& opt) {
  BucketPlan pl;
  pl.n = n;
  pl.cap2 = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(opt.bucket_cap, 16), DD_CAP);
  // mean final bucket = two thirds of the capacity or less (the shared-memory table then runs at <= 50 % load)
  int bits = 2;
  while (bits < 18 && (n >> bits) > (uint64_t)pl.cap2 * 2 / 3) ++bits;
  pl.b1 = (bits + 1) / 2;
  pl.b2 = bits - pl.b1;
  const uint64_t mean1 = ceil_div(n, 1ull << pl.b1);
  pl.cap1 = (uint32_t)((mean1 + mean1 * opt.bucket_slack_permille / 1000 + opt.bucket_headroom + 3) & ~3ull);
  pl.usable = (n >> bits) <= (uint64_t)pl.cap2 * 2 / 3 && n < (1ull << 29);
  pl.partition_threads = (int)opt.partition_threads;
  pl.dedup_threads = (int)opt.dedup_threads;
  return pl;
}

template <int T>
static int launch_partitions(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& pl, const uint32_t* cur, uint32_t n_cur, uint32_t n_next,
                             const uint32_t* child_first, const uint32_t* child_multi, uint32_t* aux, uint32_t* first_bits, uint32_t* multi_bits,
                             uint32_t* count1, uint32_t* count2, uint32_t* overflow, const LeafFinish* leaf) {
  cudaStream_t st = ctx.stream;
  constexpr int TILE = T * PT_ITEMS;
  const size_t smem = pt_smem(T);
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_leaves_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_kernel<true, T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_kernel<false, T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (leaf) {
    Launch l(ctx, "bucket_partition");
    partition_leaves_kernel<T><<<(unsigned)ceil_div(n_next, TILE), T, smem, st>>>(*leaf, n_cur, n_next, ws.keys1.ptr, ws.pos1.ptr, count1, pl.cap1, 64 - pl.b1,
                                                                               pl.b1, aux, first_bits, multi_bits, overflow, 0u);
  } else {
    Launch l(ctx, "bucket_partition");
    partition_kernel<true, T, false><<<(unsigned)ceil_div(n_next, TILE), T, smem, st>>>(
        cur, n_cur, n_next, nullptr, nullptr, nullptr, 0u, ws.keys1.ptr, ws.pos1.ptr, count1, pl.cap1, 64 - pl.b1, pl.b1, aux, first_bits, multi_bits,
        child_first, child_multi, overflow, 1u, 0u, PeerDest{});
  }
  {
    Launch l(ctx, "bucket_partition");
    const dim3 grid((unsigned)ceil_div(pl.cap1, TILE), 1u << pl.b1);
    partition_kernel<false, T, false><<<grid, T, smem, st>>>(nullptr, 0u, 0u, ws.keys1.ptr, ws.pos1.ptr, count1, pl.cap1, ws.keys2.ptr, ws.pos2.ptr,
                                                             count2, pl.cap2, 64 - pl.b1 - pl.b2, pl.b2, nullptr, nullptr, nullptr, nullptr, nullptr, overflow + 1,
                                                             1u, 0u, PeerDest{});
  }
  return STB_OK;
}

// What runs when a final bucket outgrew its region (device-side decision: all three return at once otherwise).
template <int T, int D>
static int launch_exact_pass(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& pl, uint32_t nb, const uint32_t* count1, uint32_t* count2, uint32_t* exact_off,
                             uint32_t* aux, uint32_t* first_bits, uint32_t* multi_bits, uint32_t* overflow) {
  cudaStream_t st = ctx.stream;
  const size_t smem = pt_smem(T);
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_exact_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  STB_CUDA(ctx, cudaFuncSetAttribute(bucket_dedup_chunked_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DD_SMEM));
  Launch l(ctx, "bucket_exact");
  exact_offsets_kernel<<<1, 1024, 0, st>>>(count2, nb, exact_off, overflow);
  const uint32_t tiles_x = (uint32_t)ceil_div(pl.cap1, T * PT_ITEMS), tiles_y = 1u << pl.b1;
  partition_exact_kernel<T><<<(unsigned)std::min<uint64_t>((uint64_t)tiles_x * tiles_y, 148 * (2048 / T)), T, smem, st>>>(
      ws.keys1.ptr, ws.pos1.ptr, count1, pl.cap1, ws.keys2.ptr, ws.pos2.ptr, count2, 64 - pl.b1 - pl.b2, pl.b2, overflow, exact_off, tiles_x, tiles_y);
  STB_CUDA(ctx, cudaFuncSetAttribute(bucket_dedup_kernel<D, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DD_SMEM));
  bucket_dedup_kernel<D, false, true><<<nb, D, DD_SMEM, st>>>(ws.keys2.ptr, ws.pos2.ptr, exact_off, 0u, aux, first_bits, multi_bits, overflow, PeerHome{});
  bucket_dedup_chunked_kernel<D><<<std::min<uint32_t>(nb, 148 * 4), D, DD_SMEM, st>>>(ws.keys2.ptr, ws.pos2.ptr, exact_off, nb, aux, first_bits, multi_bits,
                                                                                      overflow);
  return STB_OK;
}

template <int T>
static int launch_dedup(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& pl, uint32_t nb, const uint32_t* count2, uint32_t* aux, uint32_t* first_bits,
                        uint32_t* multi_bits, const uint32_t* overflow) {
  STB_CUDA(ctx, cudaFuncSetAttribute(bucket_dedup_kernel<T, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DD_SMEM));
  Launch l(ctx, "bucket_dedup");
  bucket_dedup_kernel<T, false><<<nb, T, DD_SMEM, ctx.stream>>>(ws.keys2.ptr, ws.pos2.ptr, count2, pl.cap2, aux, first_bits, multi_bits, overflow,
                                                               PeerHome{});
  return STB_OK;
}

// ---- sharded build (shard.cu drives these) ---------------------------------------------------
constexpr int SH_PT = 512, SH_DD = 512;

// Step 1 of a sharded level: this rank's positions -> records in its own first-pass buckets (the owners pull them).
int shard_partition(Ctx& ctx, const ShardBuckets& sb, const uint32_t* cur, uint32_t n_cur, uint32_t n_next, uint32_t pos_base,
                    const uint32_t* child_first, const uint32_t* child_multi, uint32_t* aux, uint32_t* first_bits, uint32_t* multi_bits,
                    unsigned long long* seg_keys, uint32_t* seg_pos, uint32_t* seg_count, uint32_t* overflow, const LeafFinish* leaf) {
  const size_t smem = pt_smem(SH_PT);
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_kernel<true, SH_PT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_leaves_kernel<SH_PT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (n_next == 0) return STB_OK;
  Launch l(ctx, "shard_partition");
  if (leaf) {  // the first node level: the leaf words are finished on the way
    partition_leaves_kernel<SH_PT><<<(unsigned)ceil_div(n_next, SH_PT * PT_ITEMS), SH_PT, smem, ctx.stream>>>(
        *leaf, n_cur, n_next, seg_keys, seg_pos, seg_count, sb.cap_seg, 64 - sb.b1, sb.b1, aux, first_bits, multi_bits, overflow, pos_base);
    return STB_OK;
  }
  partition_kernel<true, SH_PT, false><<<(unsigned)ceil_div(n_next, SH_PT * PT_ITEMS), SH_PT, smem, ctx.stream>>>(
      cur, n_cur, n_next, nullptr, nullptr, nullptr, 0u, seg_keys, seg_pos, seg_count, sb.cap_seg, 64 - sb.b1, sb.b1, aux, first_bits, multi_bits,
      child_first, child_multi, overflow, 1u, pos_base, PeerDest{});
  return STB_OK;
}

// Step 2 (owner): every rank's segments for this owner -> final buckets -> dedup; the answers go into per-home lists.
int shard_dedup(Ctx& ctx, const ShardBuckets& sb, BucketWorkspace& ws, uint32_t* count2, uint32_t* overflow) {
  cudaStream_t st = ctx.stream;
  const size_t smem = pt_smem(SH_PT);
  STB_CUDA(ctx, cudaFuncSetAttribute(partition_kernel<false, SH_PT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  STB_CUDA(ctx, cudaFuncSetAttribute(bucket_dedup_kernel<SH_DD, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DD_SMEM));
  const uint32_t local1 = 1u << sb.dest.bucket_shift;  // first-pass buckets this rank owns
  const uint32_t nb = local1 << sb.b2;
  STB_CUDA(ctx, ws.keys2.ensure((uint64_t)nb * sb.cap2, st));
  STB_CUDA(ctx, ws.pos2.ensure((uint64_t)nb * sb.cap2, st));
  STB_CUDA(ctx, cudaMemsetAsync(count2, 0, (uint64_t)nb * 4, st));
  {
    Launch l(ctx, "shard_partition2");
    const dim3 grid((unsigned)ceil_div(sb.cap_seg, SH_PT * PT_ITEMS), local1 * sb.dest.world);
    partition_kernel<false, SH_PT, true><<<grid, SH_PT, smem, st>>>(nullptr, 0u, 0u, nullptr, nullptr, nullptr, sb.cap_seg, ws.keys2.ptr, ws.pos2.ptr, count2,
                                                                    sb.cap2, 64 - sb.b1 - sb.b2, sb.b2, nullptr, nullptr, nullptr, nullptr, nullptr, overflow,
                                                                    sb.dest.world, 0u, sb.dest);
  }
  {
    Launch l(ctx, "shard_dedup");
    bucket_dedup_kernel<SH_DD, true><<<nb, SH_DD, DD_SMEM, st>>>(ws.keys2.ptr, ws.pos2.ptr, count2, sb.cap2, nullptr, nullptr, nullptr, overflow, sb.home);
  }
  return STB_OK;
}

int bucket_reserve(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& pl) {
  cudaStream_t st = ctx.stream;
  const uint64_t r1 = (uint64_t)pl.cap1 << pl.b1, r2 = (uint64_t)pl.cap2 << (pl.b1 + pl.b2);
  STB_CUDA(ctx, ws.keys1.ensure(r1, st));
  STB_CUDA(ctx, ws.pos1.ensure(r1, st));
  STB_CUDA(ctx, ws.keys2.ensure(r2, st));
  STB_CUDA(ctx, ws.pos2.ensure(r2, st));
  // counts of both passes, the two overflow words, the exact-size offsets (one more than there are final buckets)
  STB_CUDA(ctx, ws.counters.ensure((1ull << pl.b1) + 2 * (1ull << (pl.b1 + pl.b2)) + 4, st));
  return STB_OK;
}

int bucket_dedup_level(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& pl, const uint32_t* cur, uint32_t n_cur, uint32_t n_next,
                       const uint32_t* child_first, const uint32_t* child_multi, uint32_t* aux, uint32_t* first_bits, uint32_t* multi_bits,
                       uint32_t** overflow_out, const LeafFinish* leaf) {
  cudaStream_t st = ctx.stream;
  STB_TRY(bucket_reserve(ctx, ws, pl));
  const uint32_t nb1 = 1u << pl.b1, nb = 1u << (pl.b1 + pl.b2);
  uint32_t* count1 = ws.counters.ptr;
  uint32_t* count2 = count1 + nb1;
  uint32_t* overflow = count2 + nb;  // two words (see exact_pass_wanted)
  uint32_t* exact_off = overflow + 2;
  STB_CUDA(ctx, cudaMemsetAsync(ws.counters.ptr, 0, ((uint64_t)nb1 + nb + 2) * 4, st));
  if (pl.partition_threads == 512)
    STB_TRY(launch_partitions<512>(ctx, ws, pl, cur, n_cur, n_next, child_first, child_multi, aux, first_bits, multi_bits, count1, count2, overflow, leaf));
  else
    STB_TRY(launch_partitions<1024>(ctx, ws, pl, cur, n_cur, n_next, child_first, child_multi, aux, first_bits, multi_bits, count1, count2, overflow, leaf));
  if (pl.dedup_threads == 256) STB_TRY(launch_dedup<256>(ctx, ws, pl, nb, count2, aux, first_bits, multi_bits, overflow));
  else if (pl.dedup_threads == 512) STB_TRY(launch_dedup<512>(ctx, ws, pl, nb, count2, aux, first_bits, multi_bits, overflow));
  else STB_TRY(launch_dedup<1024>(ctx, ws, pl, nb, count2, aux, first_bits, multi_bits, overflow));
  if (pl.partition_threads == 512) STB_TRY((launch_exact_pass<512, 512>(ctx, ws, pl, nb, count1, count2, exact_off, aux, first_bits, multi_bits, overflow)));
  else STB_TRY((launch_exact_pass<1024, 512>(ctx, ws, pl, nb, count1, count2, exact_off, aux, first_bits, multi_bits, overflow)));
  *overflow_out = overflow;
  return STB_OK;
}

}  // namespace stb
