// common.cuh — device helpers and host context shared by every translation unit.
//
// Semantics follow SURVEY.md Appendix A (derived from, and verified against, the
// reference: include/dna.h, src/dna.cpp, include/shared_tree.h,
// src/shared_tree.cpp).  Nothing here is translated from the reference's code:
// the reference loops over nucleotides and builds tuples; these are closed-form
// bit manipulations on the raw 64-bit leaf / 32-bit pointer words.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/shared_tree_b200.h"

namespace stb {

// ---- raw pointer layout (reference include/shared_tree.h:73-76) -------------------
constexpr uint32_t IDX_MASK = 0x1fffffffu;
constexpr uint32_t MIRROR = 0x20000000u;
constexpr uint32_t TRANSPOSE = 0x40000000u;
constexpr uint32_t INVARIANT = 0x80000000u;
constexpr uint32_t KEY31 = 0x7fffffffu;
constexpr uint32_t PTR_NULL = 0x9fffffffu;
constexpr unsigned long long EMPTY_KEY = 0xffffffffffffffffull;

// direct leaf mode: a per-position word with this bit names a slot of the side table (a leaf with
// symbols outside ACGT) instead of a 2-bit code of the direct table (codes are below 2^24)
constexpr uint32_t LEAF_SIDE = 1u << 28;

// pointer{index, m, t, inv} (reference src/shared_tree.cpp:86-87).  `flags` carries
// m/t/inv already at bits 29/30/31; the mirror bit is dropped on invariant targets.
__host__ __device__ __forceinline__ uint32_t finish_pointer(uint32_t index, uint32_t flags) {
  const uint32_t inv = flags & INVARIANT;
  const uint32_t m = (flags & MIRROR) & ~(inv >> 2);
  return index | m | (flags & TRANSPOSE) | inv;
}

// pointer{p, m, t} (reference src/shared_tree.cpp:76-80); m, t in {0,1}.
__host__ __device__ __forceinline__ uint32_t compose(uint32_t p, uint32_t m, uint32_t t) {
  const uint32_t inv = p >> 31;
  const uint32_t is_null = ((p & KEY31) == IDX_MASK) ? 1u : 0u;
  const uint32_t nm = (m ^ ((p >> 29) & 1u)) & (inv ^ 1u);
  const uint32_t nt = (t ^ ((p >> 30) & 1u)) & (is_null ^ 1u);
  return (p & (IDX_MASK | INVARIANT)) | (nm << 29) | (nt << 30);
}

__host__ __device__ __forceinline__ bool ptr_is_null(uint32_t p) { return (p & KEY31) == IDX_MASK; }

__host__ __device__ __forceinline__ unsigned long long pair_key(uint32_t l, uint32_t r) {
  return ((unsigned long long)(l & KEY31) << 32) | (unsigned long long)(r & KEY31);
}

// node::canonical + emplace_node's invariant (reference include/shared_tree.h:115-126,
// src/shared_tree.cpp:662-672).  Returns the canonical children; flags at bits 29..31.
// For the pointers this library makes (finish_pointer, PTR_NULL: mirror never set on an invariant
// target) compose() with constant arguments is an XOR: transposing flips bit 30 unless the
// pointer is null, mirroring flips bit 29 unless the target is invariant.  The four variants are
// compared on their 31-bit keys, in the reference's order of preference (identity, transposed,
// mirrored, inverted: variadic_min keeps the first minimum, utility.h:164-170).
__host__ __device__ __forceinline__ void canonical_node(uint32_t l, uint32_t r, uint32_t& cl, uint32_t& cr,
                                                        uint32_t& flags) {
  const uint32_t tl = ptr_is_null(l) ? 0u : TRANSPOSE, tr = ptr_is_null(r) ? 0u : TRANSPOSE;
  const uint32_t ml = (~l >> 2) & MIRROR, mr = (~r >> 2) & MIRROR;
  const uint32_t lt = l ^ tl, rt = r ^ tr, lm = l ^ ml, rm = r ^ mr;
  unsigned long long best = pair_key(l, r);
  cl = l;
  cr = r;
  flags = 0;
  unsigned long long k = pair_key(lt, rt);  // (m,t) = (0,1)
  if (k < best) { best = k; cl = lt; cr = rt; flags = TRANSPOSE; }
  k = pair_key(rm, lm);                     // (1,0)
  if (k < best) { best = k; cl = rm; cr = lm; flags = MIRROR; }
  k = pair_key(rm ^ tr, lm ^ tl);           // (1,1)
  if (k < best) { best = k; cl = rm ^ tr; cr = lm ^ tl; flags = MIRROR | TRANSPOSE; }
  if ((l & KEY31) == (rm & KEY31)) flags |= INVARIANT;
}

// ---- leaves (reference src/dna.cpp:104-143) -----------------------------------------
__host__ __device__ __forceinline__ unsigned long long leaf_transposed(unsigned long long v) {
  v = ((v >> 1) & 0x5555555555555555ull) | ((v & 0x5555555555555555ull) << 1);
  v = ((v >> 2) & 0x3333333333333333ull) | ((v & 0x3333333333333333ull) << 2);
  return v;
}

__host__ __device__ __forceinline__ unsigned long long bit_reverse64(unsigned long long v) {
#ifdef __CUDA_ARCH__
  return __brevll(v);
#else
  v = ((v >> 1) & 0x5555555555555555ull) | ((v & 0x5555555555555555ull) << 1);
  v = ((v >> 2) & 0x3333333333333333ull) | ((v & 0x3333333333333333ull) << 2);
  v = ((v >> 4) & 0x0f0f0f0f0f0f0f0full) | ((v & 0x0f0f0f0f0f0f0f0full) << 4);
  v = ((v >> 8) & 0x00ff00ff00ff00ffull) | ((v & 0x00ff00ff00ff00ffull) << 8);
  v = ((v >> 16) & 0x0000ffff0000ffffull) | ((v & 0x0000ffff0000ffffull) << 16);
  return (v >> 32) | (v << 32);
#endif
}

// inverted = mirrored(transposed(x)): a full 64-bit reversal reverses both the nibble
// order and the bits inside each nibble.
__host__ __device__ __forceinline__ unsigned long long leaf_inverted(unsigned long long v, int S) {
  return bit_reverse64(v) >> (64 - 4 * S);
}
__host__ __device__ __forceinline__ unsigned long long leaf_mirrored(unsigned long long v, int S) {
  return leaf_transposed(leaf_inverted(v, S));
}

// dna::canonical: minimum over (value, mirror, transpose); flags at bits 29..31.
__host__ __device__ __forceinline__ unsigned long long canonical_leaf(unsigned long long v, int S, uint32_t& flags) {
  const unsigned long long t = leaf_transposed(v);
  const unsigned long long i = leaf_inverted(v, S);
  const unsigned long long m = leaf_transposed(i);
  unsigned long long best = v;
  flags = 0;
  if (t < best) { best = t; flags = TRANSPOSE; }
  if (m < best) { best = m; flags = MIRROR; }
  if (i < best) { best = i; flags = MIRROR | TRANSPOSE; }
  if (v == m) flags |= INVARIANT;
  return best;
}

__host__ __device__ __forceinline__ unsigned long long leaf_mask(int S) {
  return S >= 16 ? ~0ull : ((1ull << (4 * S)) - 1ull);
}

// True when every one of the S nibbles is A/C/G/T (one-hot).
__host__ __device__ __forceinline__ bool leaf_is_acgt(unsigned long long v, int S) {
  const unsigned long long ones = 0x1111111111111111ull;
  const unsigned long long pop = (v & ones) + ((v >> 1) & ones) + ((v >> 2) & ones) + ((v >> 3) & ones);
  return pop == (ones & leaf_mask(S));
}

// One-hot 4-bit codes (A1 C2 G4 T8) -> 2-bit codes (A0 C1 G2 T3), nucleotide i at bits 2i.
// Order-isomorphic to the 4-bit form, so canonical(4-bit) maps to the same class.
__host__ __device__ __forceinline__ uint32_t leaf_to_2bit(unsigned long long v) {
  const unsigned long long ones = 0x1111111111111111ull;
  const unsigned long long b = (v >> 1) & ones, c = (v >> 2) & ones, d = (v >> 3) & ones;
  unsigned long long x = b | (c << 1) | d | (d << 1);
  x = (x | (x >> 2)) & 0x0f0f0f0f0f0f0f0full;
  x = (x | (x >> 4)) & 0x00ff00ff00ff00ffull;
  x = (x | (x >> 8)) & 0x0000ffff0000ffffull;
  x = (x | (x >> 16)) & 0x00000000ffffffffull;
  return (uint32_t)x;
}

__host__ __device__ __forceinline__ unsigned long long leaf_from_2bit(uint32_t code, int S) {
  unsigned long long x = code;
  x = (x | (x << 16)) & 0x0000ffff0000ffffull;
  x = (x | (x << 8)) & 0x00ff00ff00ff00ffull;
  x = (x | (x << 4)) & 0x0f0f0f0f0f0f0f0full;
  x = (x | (x << 2)) & 0x3333333333333333ull;
  const unsigned long long ones = 0x1111111111111111ull;
  const unsigned long long lo = x & ones, hi = (x >> 1) & ones;
  const unsigned long long v = (~lo & ~hi & ones) | ((lo & ~hi) << 1) | ((~lo & hi) << 2) | ((lo & hi) << 3);
  return v & leaf_mask(S);
}

// ---- hashing -----------------------------------------------------------------------
__host__ __device__ __forceinline__ unsigned long long mix64(unsigned long long k) {
  k ^= k >> 33;
  k *= 0xff51afd7ed558ccdull;
  k ^= k >> 33;
  k *= 0xc4ceb9fe1a85ec53ull;
  return k;
}
__host__ __device__ __forceinline__ uint32_t hash64(unsigned long long k) { return (uint32_t)(mix64(k) >> 32); }

// 16-byte open-addressing slot, claimed whole by one 128-bit CAS.  `minpos` is the
// smallest level position that produced the key (atomicMin afterwards).  The last word
// is padding: ids are never stored in the table (see resolve_kernel).
struct __align__(16) Slot {
  unsigned long long key;
  uint32_t minpos;
  uint32_t pad;
};

#ifdef __CUDACC__
__device__ __forceinline__ void load_slot(const Slot* s, unsigned long long& key, uint32_t& minpos) {
  // two single-copy-atomic 64-bit elements, read at L2 (the point of coherence for the CAS)
  unsigned long long a, b;
  asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(s));
  key = a;
  minpos = (uint32_t)b;
}

// 128-bit compare-and-swap on a whole slot (sm_90+: atom.cas.b128).  Claims an empty
// slot with key AND min-position in one L2 atomic; returns the previous contents.
__device__ __forceinline__ void claim_slot(Slot* s, unsigned long long key, uint32_t pos, unsigned long long& old_key,
                                           uint32_t& old_minpos) {
  const unsigned long long empty = EMPTY_KEY;
  const unsigned long long hi = 0xffffffff00000000ull | pos;
  unsigned long long olo, ohi;
  asm volatile(
      "{\n\t"
      ".reg .b128 cmp, val, old;\n\t"
      "mov.b128 cmp, {%2, %2};\n\t"
      "mov.b128 val, {%3, %4};\n\t"
      "atom.global.cas.b128 old, [%5], cmp, val;\n\t"
      "mov.b128 {%0, %1}, old;\n\t"
      "}"
      : "=l"(olo), "=l"(ohi)
      : "l"(empty), "l"(key), "l"(hi), "l"(s)
      : "memory");
  old_key = olo;
  old_minpos = (uint32_t)ohi;
}

// Finds or claims the slot of `key` and lowers its min-position to `pos`.
// PROBE_FIRST: read the slot before trying to claim it (levels where most positions
// repeat an earlier key); otherwise claim optimistically (levels where most keys are
// new: one atomic per position instead of load + CAS + min).
// Slot `cap` (one past the probed range) is reserved for the key that equals the
// empty marker (only the 16-nucleotide leaf "----------------" can).
// First-occurrence bookkeeping without a second pass: whoever becomes a key's minimum toggles
// its own bit, and toggles the bit of the position it displaced.  XOR commutes, so whatever
// order those two atomics land in, a bit ends up set iff its position became the minimum and
// was never displaced - i.e. iff it is the key's first occurrence.
__device__ __forceinline__ void toggle_bit(uint32_t* bits, uint32_t pos) { atomicXor(bits + (pos >> 5), 1u << (pos & 31)); }

// Probing starts at slot `s`; after `limit` occupied slots it restarts once at `s_alt` (callers
// that place keys by locality use this to escape a crowded neighbourhood).  `first_bits`
// (optional) is the level's first-occurrence bitmap, maintained as described above.
template <bool PROBE_FIRST>
__device__ __forceinline__ uint32_t table_insert_from(Slot* tab, uint32_t cap, unsigned long long key, uint32_t pos, uint32_t s,
                                                      uint32_t* first_bits = nullptr, uint32_t s_alt = 0,
                                                      uint32_t limit = 0xffffffffu) {
  uint32_t steps = 0;
  if (key == EMPTY_KEY) {
    s = cap;
    if (__ldcg(&tab[s].minpos) <= pos) return s;
  } else {
    for (;;) {
      unsigned long long k;
      uint32_t mp;
      bool probed = false;
      if (PROBE_FIRST) {
        load_slot(tab + s, k, mp);
        probed = (k != EMPTY_KEY);
      }
      if (!probed) {
        claim_slot(tab + s, key, pos, k, mp);
        if (k == EMPTY_KEY) {  // claimed: key and min-position written together
          if (first_bits) toggle_bit(first_bits, pos);
          return s;
        }
      }
      if (k == key) {
        if (mp <= pos) return s;  // min-position only ever decreases
        break;
      }
      if (++steps == limit) s = s_alt;
      else if (++s == cap) s = 0;
    }
  }
  const uint32_t old = atomicMin(&tab[s].minpos, pos);
  if (first_bits && old > pos) {
    toggle_bit(first_bits, pos);
    if (old != 0xffffffffu) toggle_bit(first_bits, old);
  }
  return s;
}

template <bool PROBE_FIRST>
__device__ __forceinline__ uint32_t table_insert(Slot* tab, uint32_t cap, unsigned long long key, uint32_t pos,
                                                 uint32_t* first_bits = nullptr) {
  return table_insert_from<PROBE_FIRST>(tab, cap, key, pos, __umulhi(hash64(key), cap), first_bits);
}

// 128-bit CAS with an arbitrary expected value; returns the previous contents.
__device__ __forceinline__ void cas_slot(Slot* s, unsigned long long exp_lo, unsigned long long exp_hi, unsigned long long new_lo,
                                         unsigned long long new_hi, unsigned long long& old_lo, unsigned long long& old_hi) {
  asm volatile(
      "{\n\t"
      ".reg .b128 cmp, val, old;\n\t"
      "mov.b128 cmp, {%2, %3};\n\t"
      "mov.b128 val, {%4, %5};\n\t"
      "atom.global.cas.b128 old, [%6], cmp, val;\n\t"
      "mov.b128 {%0, %1}, old;\n\t"
      "}"
      : "=l"(old_lo), "=l"(old_hi)
      : "l"(exp_lo), "l"(exp_hi), "l"(new_lo), "l"(new_hi), "l"(s)
      : "memory");
}

// Node-level insert into an epoch-tagged table: a slot whose last word is not `serial` is stale
// (left by an earlier level), i.e. empty; it is claimed by a 128-bit CAS against exactly what was
// read, writing key, min-position and tag at once.  Probing starts at `s`; after `limit` occupied
// slots it restarts once at `s_alt`.  Keeps the first-occurrence bitmap current (toggle_bit).
__device__ __forceinline__ uint32_t tagged_insert(Slot* tab, uint32_t cap, unsigned long long key, uint32_t pos, uint32_t serial,
                                                  uint32_t s, uint32_t s_alt, uint32_t limit, uint32_t* first_bits) {
  const unsigned long long fresh_hi = ((unsigned long long)serial << 32) | pos;
  uint32_t steps = 0;
  for (;;) {
    unsigned long long k, w;
    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(k), "=l"(w) : "l"(tab + s));
    if ((uint32_t)(w >> 32) != serial) {
      unsigned long long ok, ow;
      cas_slot(tab + s, k, w, key, fresh_hi, ok, ow);
      if (ok == k && ow == w) {
        toggle_bit(first_bits, pos);
        return s;
      }
      k = ok;
      w = ow;  // somebody else claimed it in this epoch
    }
    if (k == key) {
      if ((uint32_t)w > pos) {
        const uint32_t old = atomicMin(&tab[s].minpos, pos);
        if (old > pos) {
          toggle_bit(first_bits, pos);
          toggle_bit(first_bits, old);
        }
      }
      return s;
    }
    if (++steps == limit) s = s_alt;
    else if (++s == cap) s = 0;
  }
}
#endif

// ---- host context ------------------------------------------------------------------
struct Ctx {
  int device = 0;
  int S = 12;
  cudaStream_t stream = nullptr;
  mutable std::string error;
  bool profiling = false;
  int profile_level = -1;  // >= 0: launches are accounted per level ("name@L<level>"; option profile_levels)

  struct Pending { const char* name; cudaEvent_t a, b; int level; };
  std::vector<Pending> pending;
  std::vector<cudaEvent_t> event_pool;
  struct Acc { double ms = 0; uint64_t launches = 0; };
  std::map<std::string, Acc> acc;
  std::vector<std::string> acc_order;

  int fail(int status, const std::string& msg) const {
    error = msg;
    return status;
  }
  int fail_cuda(cudaError_t e, const char* what, const char* file, int line) const {
    error = std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + file + ":" + std::to_string(line) + " (" + what + ")";
    return STB_ERR_CUDA;
  }
  cudaEvent_t get_event();
  void flush_profile();  // synchronises and folds pending events into acc
  Acc& account(const char* name, int level);  // the class "name" (level >= 0: "name@L<level>") in acc
  // a second stream for chunked host-to-device copies that later work on `stream` waits for chunk by chunk
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> copy_events;
  cudaError_t copy_lane(size_t events);
  ~Ctx();
};

extern uint64_t g_kernel_launches;

// RAII timing scope around one kernel launch (or one memset / copy).
struct Launch {
  Ctx& ctx;
  Ctx::Pending p{};
  bool kernel;
  Launch(Ctx& c, const char* name, bool is_kernel = true) : ctx(c), kernel(is_kernel) {
    if (kernel) ++g_kernel_launches;
    if (ctx.profiling) {
      p.name = name;
      p.level = ctx.profile_level;
      p.a = ctx.get_event();
      p.b = ctx.get_event();
      cudaEventRecord(p.a, ctx.stream);
    }
  }
  ~Launch() {
    if (ctx.profiling) {
      cudaEventRecord(p.b, ctx.stream);
      ctx.pending.push_back(p);
    }
  }
};

#define STB_CUDA(ctx, expr)                                                              \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess) return (ctx).fail_cuda(e__, #expr, __FILE__, __LINE__);      \
  } while (0)

#define STB_TRY(expr)                 \
  do {                                \
    int s__ = (expr);                 \
    if (s__ != STB_OK) return s__;    \
  } while (0)

// Stream-ordered device buffer.
template <typename T>
struct DevBuf {
  T* ptr = nullptr;
  uint64_t count = 0;
  cudaStream_t stream = nullptr;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept { *this = std::move(o); }
  DevBuf& operator=(DevBuf&& o) noexcept {
    if (this != &o) {
      release();
      ptr = o.ptr; count = o.count; stream = o.stream;
      o.ptr = nullptr; o.count = 0;
    }
    return *this;
  }
  ~DevBuf() { release(); }
  cudaError_t alloc(uint64_t n, cudaStream_t s) {
    release();
    stream = s;
    count = n;
    if (n == 0) n = 1;
    return cudaMallocAsync((void**)&ptr, n * sizeof(T), s);
  }
  // grow-only: keeps the current block when it is already large enough; *grew tells the caller
  // that the contents are new (uninitialised) memory
  cudaError_t ensure(uint64_t n, cudaStream_t s, bool* grew = nullptr) {
    if (grew) *grew = false;
    if (ptr && count >= n) return cudaSuccess;
    if (grew) *grew = true;
    return alloc(n, s);
  }
  void release() {
    if (ptr) cudaFreeAsync(ptr, stream);
    ptr = nullptr;
    count = 0;
  }
  uint64_t bytes() const { return count * sizeof(T); }
};

static inline uint64_t ceil_div(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

}  // namespace stb
