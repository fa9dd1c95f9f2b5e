// bucket.cuh — interface of the on-chip level deduplication (bucket.cu).
#pragma once

#include <algorithm>

#include "tree.h"

namespace stb {

struct BucketPlan {
  uint64_t n = 0;      // positions of the level
  int b1 = 1, b2 = 1;  // hash bits consumed by the two partition passes
  uint32_t cap1 = 0;   // records a first-pass bucket can hold
  uint32_t cap2 = 0;   // records a final bucket can hold (<= the dedup kernel's shared-memory tile)
  bool usable = false; // false: the level is too large for final buckets of cap2 records
  int partition_threads = 512, dedup_threads = 512;  // CTA shapes (Options)
};

// ---- sharded build: records and answers travel through peer-mapped memory --------------------
constexpr int STB_MAX_RANKS = 16;

// A position that repeats its predecessor makes no record: it points at the head of its run, at most one
// partition tile before it.  Only a first occurrence that close needs the resolve kernels' second look.
constexpr uint32_t COLLAPSE_WINDOW = 4096;

struct PeerDest {               // the first-pass buckets of every rank (a source keeps what it makes; owners pull)
  char* base[STB_MAX_RANKS] = {};  // the arena of every rank (own included)
  uint64_t keys_off = 0, pos_off = 0, count_off = 0;  // bucket arrays and their record counts inside an arena
  uint32_t bucket_shift = 0;    // log2(first-pass buckets per owner): bucket d belongs to rank d >> bucket_shift
  uint32_t src = 0, world = 1;  // this rank
  // the record counts of the segments this rank owns, as every source sent them (local memory:
  // counts_in[source * counts_stride + local bucket]); null: read them from the sources' arenas
  const uint32_t* counts_in = nullptr;
  uint32_t counts_stride = 0;
};

struct PeerHome {               // where the answers about a position go: a list per home rank, in the owner's arena
  char* base[STB_MAX_RANKS] = {};
  uint64_t ans_off = 0, ans_count_off = 0;
  uint32_t ans_cap = 0;         // answers one owner can hold for one home rank
  uint32_t self = 0;
  uint32_t log2_positions = 0;  // positions per rank at this level (a power of two): home = position >> log2_positions
  // how many answers every owner keeps for this rank, as the owners sent them (local: counts_in[owner * counts_stride])
  const uint32_t* counts_in = nullptr;
  uint32_t counts_stride = 0;
};

struct ShardBuckets {
  int b1 = 1, b2 = 1;           // hash bits of the two passes (the top log2(world) bits of the first choose the owner)
  uint32_t cap_seg = 0;         // records one source may send to one first-pass bucket
  uint32_t cap2 = 0;            // records of a final bucket
  PeerDest dest;
  PeerHome home;
};

// Leaf pointers finished on the fly by the first node level's partition pass (ACGT text through the direct
// leaf table).  That pass is the first kernel to hold both children of a node position, and the 258 M lookups in
// the L2-resident id table hide behind its integer work instead of being a kernel of their own (resolve<leaf>,
// 1.2 ms at 3.1 Gbp).  The pass writes the finished pointers back, so every later reader sees what resolve<leaf>
// would have left.
struct LeafFinish {
  uint32_t* words = nullptr;             // the leaf level's per-position words: finished pointers at the first occurrences,
                                         // canonical code | flags (or LEAF_SIDE | side slot | flags) everywhere else
  const uint32_t* first_bits = nullptr;  // the leaf level's first occurrences
  const uint32_t* dids = nullptr;        // id by canonical 2-bit code
  const Slot* side = nullptr;            // leaves outside ACGT: min-position per leaf (its word holds the id)
  const uint32_t* done_bits = nullptr;   // later occurrences the leaf kernel already finished (null: none)
};

struct BucketWorkspace {
  DevBuf<unsigned long long> keys1, keys2;
  DevBuf<uint32_t> pos1, pos2, counters;
};

BucketPlan bucket_plan(uint64_t n, const Options& opt);
int bucket_reserve(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& plan);

// Deduplicates the node level whose children are cur[0, n_cur): afterwards first_bits marks the
// first occurrences, aux[p] = flags(p) | position of p's first occurrence for the later occurrences
// (aux is not written for first occurrences: assign recomputes them), multi_bits marks the first occurrences whose key occurs
// again.  child_first / child_multi (optional): the child level's bitmaps; a position with a child
// that never repeats is a certified singleton and makes no record (build.cu: children_both_repeat).
// first_bits (tile-rounded) and multi_bits must be zero on entry.  *overflow_out is a
// device flag: non-zero means a bucket overflowed and nothing of the above was produced.
int bucket_dedup_level(Ctx& ctx, BucketWorkspace& ws, const BucketPlan& plan, const uint32_t* cur, uint32_t n_cur, uint32_t n_next,
                       const uint32_t* child_first, const uint32_t* child_multi, uint32_t* aux, uint32_t* first_bits, uint32_t* multi_bits, uint32_t** overflow_out,
                       const LeafFinish* leaf = nullptr);

// shard.cu drives these: see ShardBuckets.  seg_*: this rank's first-pass buckets (2^b1 x cap_seg records and
// their counts, in its arena); the owner's split reads every rank's through `dest`.
int shard_partition(Ctx& ctx, const ShardBuckets& sb, const uint32_t* cur, uint32_t n_cur, uint32_t n_next, uint32_t pos_base,
                    const uint32_t* child_first, const uint32_t* child_multi, uint32_t* aux, uint32_t* first_bits, uint32_t* multi_bits,
                    unsigned long long* seg_keys, uint32_t* seg_pos, uint32_t* seg_count, uint32_t* overflow, const LeafFinish* leaf = nullptr);
int shard_dedup(Ctx& ctx, const ShardBuckets& sb, BucketWorkspace& ws, uint32_t* count2, uint32_t* overflow);

}  // namespace stb
