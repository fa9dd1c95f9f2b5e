// tree.h — device-resident shared_tree and the internal entry points of each stage.
#pragma once

#include <memory>

#include "common.cuh"

namespace stb {

// Mirrors the reference's private members (include/shared_tree.h:232-236):
//   std::vector<std::vector<node>> nodes;  ->  layers[k].nodes (uint2 = left,right) in HBM
//   std::vector<dna> leaves;               ->  leaves (uint64) in HBM
//   pointer root;                          ->  root
struct Layer {
  DevBuf<uint2> nodes;
  uint64_t count = 0;
};

// Tunables of a handle (stb_set_option).  The defaults are what the benchmarks run; tests lower
// the thresholds so that the large-input paths run on inputs small enough for the oracle.
struct Options {
  uint64_t bucket_min = 1ull << 22;      // node levels with at least this many positions are deduplicated on chip (partition.cu)
  uint64_t bucket_levels = 1;            // ... and only the first this many node levels of a build
  uint64_t bucket_cap = 3072;            // records a final bucket may hold (<= 3072, what the dedup kernel keeps in registers)
  uint64_t partition_threads = 512;      // CTA size of the partition passes (512 or 1024; 4 records per thread)
  uint64_t dedup_threads = 512;          // CTA size of the bucket dedup kernel (256, 512 or 1024)
  uint64_t bucket_slack_permille = 125;  // head-room of a first-pass bucket over the mean ...
  uint64_t bucket_headroom = 1024;       // ... plus this many records (a first-pass bucket that still overflows sends the level to the table in HBM)
  uint64_t child_filter = 1;             // exact singleton filter from the child level's bitmaps (node levels >= 1)
  uint64_t locality = 1;                 // slot proportional to a child id above the first node layer
  uint64_t coop_max = 1ull << 20;        // levels with at most this many pointers run in one cooperative launch
  uint64_t side_table_slots = 1ull << 22; // hash-table slots for leaves outside ACGT next to the direct leaf table (half of them usable)
  uint64_t reserve_pipeline = 1;         // a build also reserves the scratch of sort_tree and decode (the compress path always sorts)
  uint64_t stream_chunk_log2 = 24;       // leaves per chunk of the streaming host build
  uint64_t stream_min_chunks = 4;        // smaller host inputs are copied and built in one shot
  uint64_t leaf_prefix_log2 = 25;        // one-shot ACGT-12 leaf level: after this many positions the ids seen so far are final and
                                         // the rest of the leaves look them up (build.cu: leaf_insert_acgt12_kernel); 0 = one window
  uint64_t profile_levels = 0;           // the kernel timings of stb_profile_read are kept per level ("name@L3")
  uint64_t fused_resolve = 1;            // node levels of the one-shot build resolve their later occurrences in the assign pass,
                                         // from a rank directory (build.cu: assign_resolve_kernel); 0 = separate resolve pass
};

struct Tree : Ctx {
  Options opt;
  bool built = false;
  uint64_t n_leaves = 0;
  DevBuf<unsigned long long> leaves;
  std::vector<Layer> layers;
  uint32_t root = PTR_NULL;
  uint64_t width = 0;

  // Build workspace (pointer arrays, tables, bitmaps: build.cu's Scratch) and the host-input
  // staging buffer.  Both are grow-only and live until stb_destroy / stb_release_workspace, so
  // repeated builds on one handle do no device allocation.
  std::shared_ptr<void> workspace;
  DevBuf<char> staging;
  // Scratch of decode (two ping-pong pointer arrays) and of sort_tree (one arena carved by
  // offsets): grow-only as well, so repeated calls on one handle allocate nothing.
  DevBuf<uint32_t> decode_a, decode_b;
  DevBuf<char> sort_arena;
  // sort_tree permutes a layer into its spare and swaps the two (no copy back, no allocation once
  // the handle has sorted a tree of this shape)
  DevBuf<unsigned long long> spare_leaves;
  std::vector<DevBuf<uint2>> spare_nodes;
  // Scratch of region extraction: per-region item bases and output offsets (decode.cu: region_plan), and the
  // region arrays of a host-memory call (t.staging carries that call's output back, so they cannot share it).
  DevBuf<unsigned long long> region_scratch;
  DevBuf<char> region_inputs;
  void release_scratch() {
    decode_a.release();
    decode_b.release();
    region_scratch.release();
    region_inputs.release();
    sort_arena.release();
    spare_leaves.release();
    spare_nodes.clear();
  }

  // serialization plan cache (per-layer byte totals), invalidated by build / sort
  bool plan_valid = false;
  uint64_t stream_bytes = 0;
  std::vector<uint64_t> layer_stream_bytes;
  std::vector<DevBuf<unsigned long long>> layer_tile_off;  // per layer: byte offset of each 1024-node tile

  void clear() {
    built = false;
    n_leaves = 0;
    leaves.release();
    layers.clear();
    root = PTR_NULL;
    width = 0;
    plan_valid = false;
    layer_tile_off.clear();
  }
};

// ingest.cu ------------------------------------------------------------------------
// FASTA text (device) -> bare body (device, newly allocated).  body_len excludes
// nothing yet (tail truncation happens at packing).
int fasta_extract_body(Ctx& ctx, const char* d_text, uint64_t len, DevBuf<char>& body, uint64_t* body_len);
// The same chunk by chunk: the text lies in one contiguous device buffer and arrives in chunks (multiples
// of 64 KiB); the automaton's state is carried on the device; the body grows in d_body.
struct FastaStream {
  std::shared_ptr<void> impl;
};
constexpr uint64_t FASTA_STREAM_ALIGN = 65536;
int fasta_stream_begin(Ctx& ctx, FastaStream& fs, uint64_t max_chunk_bytes);
int fasta_stream_chunk(Ctx& ctx, FastaStream& fs, const char* d_text_begin, uint64_t first, uint64_t len, char* d_body);
int fasta_stream_body_len(Ctx& ctx, FastaStream& fs, uint64_t* body_len);  // synchronises: body bytes produced so far
// bare body (device) -> packed leaves (device); error on unknown symbols.
int pack_body(Ctx& ctx, const char* d_body, uint64_t n_leaves, unsigned long long* d_leaves);

// build.cu -------------------------------------------------------------------------
int build_from_body(Tree& t, const char* d_body, uint64_t body_len);
int build_from_leaves(Tree& t, const unsigned long long* d_leaves, uint64_t n);
// status of a path that does not apply to this input (the caller takes another one); every stb_status is >= 0
constexpr int NOT_APPLICABLE = -1;
int build_from_host_body(Tree& t, const char* h_body, uint64_t body_len);  // streaming, or NOT_APPLICABLE: use the one-shot path
int build_from_host_fasta(Tree& t, const char* h_text, uint64_t len);      // streaming incl. body extraction, or NOT_APPLICABLE
int build_upper_levels(Tree& t, const uint32_t* d_ptrs, uint64_t n, bool at_least_one);
int dist_leaf_direct_minpos(Ctx& ctx, const char* d_body, uint64_t n_local, uint64_t gpos0, uint32_t* dminpos, uint32_t* tmp,
                            int* non_acgt);

// dist.cu --------------------------------------------------------------------------
// (entry points are extern "C", see include/shared_tree_b200_dist.h)

// sort.cu --------------------------------------------------------------------------
int histogram_layer(const Tree& t, uint64_t layer, DevBuf<uint32_t>& freq);
int histogram_u64(const Tree& t, uint64_t layer, unsigned long long* d_out);
int sort_tree(Tree& t);
int sort_reserve(Tree& t);  // the scratch a sort_tree of this tree will need (kept by the handle)

// serialize.cu ---------------------------------------------------------------------
int stream_plan(Tree& t);
int serialize_tree(Tree& t, uint8_t* d_out, uint64_t cap);
int deserialize_tree(Tree& t, const uint8_t* h_bytes, uint64_t len);

// decode.cu ------------------------------------------------------------------------
int compute_width(Tree& t);
int decode_reserve(Tree& t);  // the scratch a full decode of this tree will need (kept by the handle)
int decode_range(const Tree& t, uint64_t first, uint64_t count, unsigned long long* d_out, char* d_ascii);
int random_access(const Tree& t, const unsigned long long* d_index, uint64_t q, unsigned long long* d_out);
// stb_extract_regions in two steps on device arrays: region_plan checks every region and sizes the output
// (the scratch it leaves on the handle is what region_write reads); region_write writes it.
struct RegionPlan {
  uint64_t total_len = 0, items = 0;
  bool hull = false;  // some regions are long enough to be read from one level expansion over groups [hull_first, hull_last]
  uint64_t hull_first = 0, hull_last = 0;
};
int region_plan(const Tree& t, const unsigned long long* d_start, const unsigned long long* d_end, const uint8_t* d_strand,
                uint64_t n, RegionPlan* plan);
int region_write(const Tree& t, const unsigned long long* d_start, const unsigned long long* d_end, const uint8_t* d_strand,
                 uint64_t n, const RegionPlan& plan, char* d_out);

// synth.cu -------------------------------------------------------------------------
int synth_genome(Ctx& ctx, char* d_out, uint64_t n_bases, uint64_t first, uint64_t count, uint64_t seed,
                 uint32_t repeat_permille);

int synth_mask(Ctx& ctx, char* d_text, uint64_t first, uint64_t count, uint64_t seed);  // N runs + soft-masking over a generated text

// shared error word for unknown symbols: (byte offset << 8) | upper-cased byte
std::string unknown_symbol_message(int upper_byte);

}  // namespace stb

// the opaque handle of the C ABI
struct stb_tree : stb::Tree {};
