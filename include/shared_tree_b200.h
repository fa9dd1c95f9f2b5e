/*
 * shared_tree_b200.h — C ABI of the B200-native shared_tree hot path.
 *
 * The reference (Quinten-van-Woerkom/genome-compression) has no FFI; its
 * boundary for this path is the C++ class surface of include/shared_tree.h
 * (used by compress.cpp:183-200 and tests/test.cpp).  Each entry point below
 * names the reference member it replaces (paths relative to the reference
 * root).  Plain pointers and sizes only; one opaque handle; int status
 * returns; no exceptions cross the boundary; no hidden globals (the
 * reference's process-global dna::size(), include/dna.h:47, is an explicit
 * per-handle argument).  INTEGRATION.md shows the C++ shim a maintainer of the
 * reference would put on top (genome-compression_b200/host/).
 *
 * Raw in-memory formats (identical to the reference's, SURVEY Appendix A):
 *   leaf     uint64, nucleotide i in bits 4i..4i+3, 4-bit IUPAC codes of
 *            include/dna.h:20-32, nibbles >= dna_size are zero
 *   pointer  uint32: bits 0-28 index, 29 mirror, 30 transpose, 31 invariant;
 *            null = 0x9fffffff            (include/shared_tree.h:73-76)
 *   node     two pointers (left, right)   (include/shared_tree.h:146)
 *
 * There is no CPU fallback: every call that computes needs a CUDA device and
 * returns STB_ERR_CUDA otherwise.
 */
#ifndef SHARED_TREE_B200_H
#define SHARED_TREE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STB_ABI_VERSION 1

typedef struct stb_tree stb_tree; /* opaque */

enum stb_status {
  STB_OK = 0,
  STB_ERR_CUDA = 1,           /* CUDA runtime error or no device; see stb_last_error */
  STB_ERR_INVALID_ARG = 2,
  STB_ERR_UNKNOWN_SYMBOL = 3, /* src/dna.cpp:44-47: "Encountered unknown symbol" + exit(1) */
  STB_ERR_EMPTY = 4,          /* fewer than dna_size bases: undefined in the reference (SIGFPE) */
  STB_ERR_BUFFER_TOO_SMALL = 5,
  STB_ERR_NOT_BUILT = 6,
  STB_ERR_INDEX_CEILING = 7,  /* a layer outgrew the 29-bit index / 28-bit offset (src/shared_tree.cpp:54-67) */
  STB_ERR_BAD_LEAF = 8,       /* packed leaf with bits set at or above 4*dna_size */
  STB_ERR_OUT_OF_RANGE = 9,   /* index >= width (precondition of operator[], src/shared_tree.cpp:266) */
  STB_ERR_BAD_STREAM = 10,    /* truncated / malformed .dag bytes */
  STB_ERR_TOO_LARGE = 11      /* 2^30 or more leaf positions */
};

enum stb_memory { STB_HOST = 0, STB_DEVICE = 1 };

/* ---- lifetime: shared_tree ctor / dtor / copy (tests/test.cpp:275) ---------- */
/* dna_size replaces dna::size(n) (compress.cpp:169); valid 1..16.
 * cuda_stream: a cudaStream_t (NULL = default stream); all work of this handle is
 * enqueued there. */
int stb_create(stb_tree** out, int device, int dna_size, void* cuda_stream);
int stb_destroy(stb_tree* tree);
int stb_clone(const stb_tree* tree, stb_tree** out);
/* A handle keeps its build workspace (tables, pointer arrays, host-input staging) between
 * builds so that repeated builds allocate nothing; this gives it back early. */
int stb_release_workspace(stb_tree* tree);

/* Tunables of the build (thresholds between its code paths; DESIGN.md §4).  Defaults are the
 * measured optimum; tests lower them to push small inputs through the large-input paths.
 * Names: "bucket_min", "bucket_levels", "bucket_cap", "partition_threads", "dedup_threads", "bucket_slack_permille", "bucket_headroom", "child_filter", "locality",
 * "coop_max", "reserve_pipeline", "side_table_slots", "stream_chunk_log2", "stream_min_chunks", "leaf_prefix_log2", "profile_levels",
 * "fused_resolve".  Unknown name: STB_ERR_INVALID_ARG. */
int stb_set_option(stb_tree* tree, const char* name, uint64_t value);
int stb_get_option(const stb_tree* tree, const char* name, uint64_t* value);

/* ---- construction --------------------------------------------------------- */
/* shared_tree(fasta_reader, bool), src/shared_tree.cpp:207 + the ingest semantics
 * of src/fasta_reader.cpp:40-68: '>' / blank lines skipped, newlines removed,
 * case folded, trailing len%dna_size bases dropped.  `text` may be host or
 * device memory. */
int stb_build_from_fasta(stb_tree* tree, const char* text, uint64_t len, int memory);
/* Same, but the caller asserts the text is already the bare body (no header,
 * no newline): skips the compaction pass. */
int stb_build_from_body(stb_tree* tree, const char* body, uint64_t len, int memory);
/* shared_tree(std::vector<dna>&, bool), src/shared_tree.cpp:212 */
int stb_build_from_leaves(stb_tree* tree, const uint64_t* leaves, uint64_t count, int memory);
/* read_genome(path), src/fasta_reader.cpp:108: FASTA text -> packed leaves.
 * *count receives the leaf count; leaves (may be NULL to query) receives
 * min(*count, cap) values in `memory`. */
int stb_pack_fasta(stb_tree* tree, const char* text, uint64_t len, int text_memory, uint64_t* leaves,
                   uint64_t cap, int leaves_memory, uint64_t* count);

/* ---- queries: include/shared_tree.h:164-170 ----------------------------------- */
int stb_depth(const stb_tree* tree, uint64_t* out);                     /* depth()  */
int stb_width(const stb_tree* tree, uint64_t* out);                     /* width()  */
int stb_leaf_count(const stb_tree* tree, uint64_t* out);                /* leaf_count() */
int stb_node_count(const stb_tree* tree, uint64_t* out);                /* node_count() */
int stb_layer_count(const stb_tree* tree, uint64_t layer, uint64_t* out); /* node_count(layer) */
int stb_root(const stb_tree* tree, uint32_t* out);                      /* private member `root` */
int stb_dna_size(const stb_tree* tree, int* out);

/* access_leaf / access_node / operator<< : raw copies of the stored tables */
int stb_copy_leaves(const stb_tree* tree, uint64_t* out, uint64_t cap, int memory);
int stb_copy_layer(const stb_tree* tree, uint64_t layer, uint32_t* out_pairs, uint64_t cap_nodes, int memory);
/* histogram(layer), src/shared_tree.cpp:316: references from node layer `layer`
 * into its child layer (the leaves for layer 0). */
int stb_histogram(const stb_tree* tree, uint64_t layer, uint64_t* out, uint64_t cap, int memory);

/* ---- sort_tree, src/shared_tree.cpp:443 ---------------------------------------- */
int stb_sort_tree(stb_tree* tree);

/* ---- .dag stream: src/shared_tree.cpp:488-546 ----------------------------------- */
int stb_bytes(const stb_tree* tree, uint64_t* out);                      /* bytes() */
int stb_serialize(const stb_tree* tree, uint8_t* out, uint64_t cap, int memory, uint64_t* written);
/* deserialize from host bytes.  STB_ERR_BAD_STREAM for: a stream that ends inside the header, the leaf table or a
 * node; no leaves, a node layer of no nodes, or no node layer; a leaf table or layer too large for the pointer format;
 * a child pointer past the end of the layer below, or the null index (segment 3, offset 0xfffffff) with the mirror or
 * transpose bit set; a root that does not index the top layer; a node on the logical right edge whose children are
 * both null.  Nulls elsewhere are accepted (builds never write them; width() and decode assume there are none). */
int stb_deserialize(stb_tree* tree, const uint8_t* bytes, uint64_t len);

/* ---- decode ------------------------------------------------------------------------ */
/* shared_tree::iterator (src/shared_tree.cpp:553-614): leaves first..first+count-1
 * in sequence order, transforms applied. */
int stb_decode_leaves(const stb_tree* tree, uint64_t first, uint64_t count, uint64_t* out, int memory);
/* same, expanded to dna_size ASCII letters per leaf (operator<<(dna), src/dna.cpp:201) */
int stb_decode_ascii(const stb_tree* tree, uint64_t first, uint64_t count, char* out, int memory);
/* operator[] (src/shared_tree.cpp:268-291), batched: out[i] = tree[index[i]] */
int stb_random_access(const stb_tree* tree, const uint64_t* index, uint64_t queries, uint64_t* out, int memory);
/* Bases [start[i], end[i]) of the decoded sequence, 0-based and half-open as in BED.
 * Base b is nucleotide b % dna_size of leaf b / dna_size; valid ends are <= width() * dna_size.
 * strand[i]: 0 = as stored, 1 = reverse complement (dna::inverted, src/dna.cpp).
 * strand may be NULL, meaning all regions are forward.
 * Letters as stb_decode_ascii spells them.  Regions go back to back in input order:
 * region i starts at out[sum of the lengths of regions 0..i-1].
 * *written receives the total length.
 * start, end, strand and out all live in `memory` (device start and end: 8-byte aligned).
 * out == NULL: only *written is set.
 * cap < total: STB_ERR_BUFFER_TOO_SMALL, *written = total, out untouched.
 * Regions may overlap, come in any order, be empty or span the whole sequence.  Every region is checked
 * before anything is written: start > end, or a strand outside {0, 1}: STB_ERR_INVALID_ARG; end past the
 * sequence: STB_ERR_OUT_OF_RANGE.  n_regions == 0: STB_OK with *written = 0. */
int stb_extract_regions(const stb_tree* tree, const uint64_t* start, const uint64_t* end, const uint8_t* strand,
                        uint64_t n_regions, char* out, uint64_t cap, int memory, uint64_t* written);

/* ---- value primitives (no device needed) ------------------------------------------------
 * The very functions the kernels run (__host__ __device__), callable on the host so that the
 * arithmetic can be checked against the reference's vectors without a GPU.
 * node::canonical + emplace_node's invariant (include/shared_tree.h:115-126, src/shared_tree.cpp:662-672):
 * flags = mirror<<29 | transpose<<30 | invariant<<31. */
void stb_node_canonical(uint32_t left, uint32_t right, uint32_t* out_left, uint32_t* out_right, uint32_t* out_flags);
/* dna::canonical (src/dna.cpp:135-143); same flag layout. */
uint64_t stb_leaf_canonical(uint64_t leaf, int dna_size, uint32_t* out_flags);
/* pointer{p, mirror, transpose} (src/shared_tree.cpp:76-80) */
uint32_t stb_pointer_compose(uint32_t pointer, int mirror, int transpose);

/* ---- diagnostics ---------------------------------------------------------------------- */
const char* stb_status_string(int status);
/* Details of the last failure on this handle.  For STB_ERR_UNKNOWN_SYMBOL the
 * text is the reference's own message ("Encountered unknown symbol: ..."). */
const char* stb_last_error(const stb_tree* tree);
/* Number of CUDA kernels this library launched in this process so far. */
uint64_t stb_kernel_launches(void);

/* Per-kernel device timing (CUDA events on the handle's stream).  Off by default. */
int stb_profile_enable(stb_tree* tree, int on);
int stb_profile_reset(stb_tree* tree);
/* Fills names[i] (static strings), total_ms[i], launches[i] for up to cap kernel
 * classes; *count receives the number of classes.
 * A level's ids: count_firsts, then assign_ids and resolve_ids; node levels built one kernel at a time
 * with the option fused_resolve (default) run tile_bases and assign_resolve instead of the last two.
 * Besides the kernels, five classes with total_ms = 0 count the on-chip (bucketed) node levels of the
 * builds profiled, one per level, by what that level's deduplication came to:
 *   dedup_on_chip              every final bucket fitted its region
 *   dedup_exact                a final bucket outgrew its region: the exact-size second pass ran
 *   dedup_chunked              ... and a final bucket of more than 3072 records was walked in chunks
 *   dedup_fallback_first_pass  a first-pass bucket overflowed: the level went through the table in HBM
 *   dedup_fallback_distinct    a chunked bucket held more than 4096 distinct keys: the same fallback
 * With the option profile_levels they carry "@L<level>" like the kernels. */
int stb_profile_read(stb_tree* tree, const char** names, double* total_ms, uint64_t* launches,
                     uint64_t cap, uint64_t* count);

/* ---- synthetic workload (bench / tests; DESIGN.md §6) -------------------------------- */
/* Fills device memory `out` with bases [first, first+count) of the synthetic
 * genome (n_bases, seed, repeat_permille): i.i.d. ACGT plus planted repeats. */
int stb_synth_genome(int device, void* cuda_stream, char* out_device, uint64_t n_bases, uint64_t first,
                     uint64_t count, uint64_t seed, uint32_t repeat_permille);

/* The "real genome" variant: lays runs of N (about 1 % of the bases) and soft-masked lower-case stretches over
 * bases [first, first+count) of a generated text in device memory (a pure function of the position). */
int stb_synth_mask(int device, void* cuda_stream, char* text_device, uint64_t first, uint64_t count, uint64_t seed);

#ifdef __cplusplus
}
#endif
#endif /* SHARED_TREE_B200_H */
