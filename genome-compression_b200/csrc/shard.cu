// shard.cu — the sharded multi-GPU build behind ONE C-ABI call per rank (BASELINE.json config 4).
//
// The reference builds a tree with one call (tree_constructor::reduce, src/shared_tree.cpp:719-736);
// so does a rank here: stb_shard_build_from_body.  One process per GPU, NCCL for the set-up and the
// leaf level (communicator, exchange of the IPC handles, the leaf table's all-reduce), peer-mapped
// memory over NVLink for everything inside the level loop: the owners pull a level's records from the
// ranks that made them, the home ranks pull the owners' answers, a later occurrence reads the id of
// its first occurrence from the home rank's pointer array, and the four synchronisation points of a
// level are one tiny kernel each (peer_exchange_kernel: a few numbers and an epoch flag stored into
// every peer's arena).  Nothing is read by the host inside the level loop.
//
// Rank g owns a contiguous, power-of-two aligned range of positions at every sharded level (the
// analogue of the reference's own 2^22 / 2^25-leaf segments, include/shared_tree.h:305-316), so
// both children of a node position are on one rank.  Ids stay first-occurrence ranks in GLOBAL
// position order - rank g's first occurrences take the ids after those of ranks 0..g-1 - so the
// gathered tree is byte-identical to the single-GPU tree and to the reference's.
//
// Per node level (every per-level cost is O(level / world) on a rank):
//   partition   local positions -> (key, global position) records, grouped by first-pass bucket in
//               shared memory, kept in this rank's arena (bucket.cu)
//   exchange    barrier + the segments' record counts to their owners
//   dedup       the owner pulls its segments from every rank, splits them into final buckets and
//               deduplicates each in shared memory; the answers (a later occurrence and where its key
//               came first; a first occurrence whose key came again) go into one list per home rank
//   exchange    barrier + the lists' lengths to the home ranks
//   apply       the home rank pulls its lists and updates its own words
//   ids         local counts; exchange: barrier + everybody's count; local assignment
//   exchange    barrier
//   resolve     later occurrences fetch the finished pointer of their first occurrence (peer load)
// Levels of at most `cut` positions are gathered on rank 0 and finished by the single-GPU code.
#include <dlfcn.h>
#include <nccl.h>

#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/shared_tree_b200_dist.h"
#include "bucket.cuh"
#include "level.cuh"
#include "tree.h"

namespace stb {

namespace {

// ---- NCCL, resolved at run time (the library loads without it; torch's copy is reused when present) ----
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
  std::string why;
};

const NcclApi& nccl() {
  static NcclApi api = [] {
    NcclApi a;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      a.why = "libnccl.so.2 not found";
      return a;
    }
    auto sym = [&](const char* name) { return dlsym(h, name); };
    a.GetUniqueId = (decltype(a.GetUniqueId))sym("ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))sym("ncclCommInitRank");
    a.CommDestroy = (decltype(a.CommDestroy))sym("ncclCommDestroy");
    a.AllReduce = (decltype(a.AllReduce))sym("ncclAllReduce");
    a.AllGather = (decltype(a.AllGather))sym("ncclAllGather");
    a.Send = (decltype(a.Send))sym("ncclSend");
    a.Recv = (decltype(a.Recv))sym("ncclRecv");
    a.GroupStart = (decltype(a.GroupStart))sym("ncclGroupStart");
    a.GroupEnd = (decltype(a.GroupEnd))sym("ncclGroupEnd");
    a.GetErrorString = (decltype(a.GetErrorString))sym("ncclGetErrorString");
    a.ok = a.GetUniqueId && a.CommInitRank && a.CommDestroy && a.AllReduce && a.AllGather && a.Send && a.Recv && a.GroupStart && a.GroupEnd;
    if (!a.ok) a.why = "libnccl.so.2 lacks a required symbol";
    return a;
  }();
  return api;
}

#define STB_NCCL(ctx, expr)                                                                                   \
  do {                                                                                                        \
    ncclResult_t r__ = (expr);                                                                                \
    if (r__ != ncclSuccess)                                                                                   \
      return (ctx).fail(STB_ERR_CUDA, std::string("NCCL error: ") + (nccl().GetErrorString ? nccl().GetErrorString(r__) : "?") + " (" #expr ")"); \
  } while (0)

__global__ void min_over_ranks_kernel(uint32_t* __restrict__ out, const uint32_t* const* __restrict__ in, int world, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    uint32_t m = 0xffffffffu;
    for (int r = 0; r < world; ++r) m = min(m, in[r][i]);
    out[i] = m;
  }
}

// ---- barrier + small all-to-all over peer-mapped memory ----------------------------------------
// A level of the sharded build needs four synchronisation points, three of which carry a few numbers
// (record counts per segment, answer counts, unique counts).  As NCCL collectives they cost 75-120 us each
// on eight GPUs, more than most of the level's kernels; here one warp per peer stores the numbers and
// then an epoch flag straight into the peer's arena over NVLink, and waits for the peers' flags in its own.
constexpr uint32_t XCHG_WORDS = 512;  // words one rank can send to one rank per exchange
constexpr int XCHG_SLOTS = 4;         // mailboxes: an exchange never overwrites what the previous three delivered

struct PeerBox {
  char* base[STB_MAX_RANKS];
  uint64_t recv_off, flag_off;
  uint32_t self, world;
};

__global__ void __launch_bounds__(STB_MAX_RANKS * 32)
peer_exchange_kernel(PeerBox box, const uint32_t* __restrict__ send, uint32_t words, uint32_t send_stride, uint32_t epoch, uint32_t* __restrict__ timeout_flag) {
  const uint32_t peer = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (peer >= box.world) return;
  uint32_t* dst = reinterpret_cast<uint32_t*>(box.base[peer] + box.recv_off) + (uint64_t)box.self * XCHG_WORDS;
  for (uint32_t i = lane; i < words; i += 32) dst[i] = send[(uint64_t)peer * send_stride + i];
  __threadfence_system();  // the numbers before the flag
  __syncwarp();
  if (lane == 0) {
    *reinterpret_cast<volatile uint32_t*>(box.base[peer] + box.flag_off + 4ull * box.self) = epoch;
    const volatile uint32_t* mine = reinterpret_cast<const volatile uint32_t*>(box.base[box.self] + box.flag_off) + peer;
    const long long t0 = clock64();
    while ((int32_t)(*mine - epoch) < 0) {
      if (clock64() - t0 > 60000000000ll) {  // a peer that never arrives (it failed on its own): give up after half a minute, not never
        *timeout_flag = 1u;
        break;
      }
    }
  }
  __threadfence_system();
}

// ---- the plumbing a rank needs ---------------------------------------------------------------
struct Comm {
  int rank = 0, world = 1;
  virtual ~Comm() {}
  virtual int barrier(Ctx& ctx) = 0;                                                  // stream-ordered: later work sees every rank's earlier work
  virtual int all_reduce_min(Ctx& ctx, uint32_t* buf, size_t n) = 0;                  // device, in place
  virtual int all_gather_u32(Ctx& ctx, const uint32_t* send, uint32_t* recv, size_t n) = 0;  // device, n words per rank
  // All-to-all of a few words + barrier, stream-ordered: `words` words starting at send + r * send_stride go to rank r, which finds
  // them at its recv + me * XCHG_WORDS; later work on the stream sees every rank's earlier work (words = 0: a plain barrier).
  // `arena` / `all`: this rank's arena and everybody's (share()); recv_off / flag_off: where the mailbox and the flags lie in an arena.
  virtual int exchange(Ctx& ctx, char* const* all, uint64_t recv_off, uint64_t flag_off, const uint32_t* send, uint32_t words, uint32_t send_stride,
                       uint32_t* timeout_flag) = 0;
  virtual int share(Ctx& ctx, char* mine, char** all) = 0;                            // peer-map every rank's arena (cudaMalloc memory)
  virtual void unshare(char** all) = 0;
  virtual int gather_to_root(Ctx& ctx, const void* send, size_t bytes, void* recv, const size_t* bytes_of) = 0;  // device, variable sizes
};

struct NcclComm : Comm {
  ncclComm_t comm = nullptr;
  DevBuf<uint32_t> token;
  DevBuf<char> hbuf;
  ~NcclComm() override {
    if (comm) nccl().CommDestroy(comm);
  }
  int barrier(Ctx& ctx) override {
    STB_CUDA(ctx, token.ensure(1, ctx.stream));
    STB_NCCL(ctx, nccl().AllReduce(token.ptr, token.ptr, 1, ncclUint32, ncclMax, comm, ctx.stream));
    return STB_OK;
  }
  int all_reduce_min(Ctx& ctx, uint32_t* buf, size_t n) override {
    STB_NCCL(ctx, nccl().AllReduce(buf, buf, n, ncclUint32, ncclMin, comm, ctx.stream));
    return STB_OK;
  }
  int all_gather_u32(Ctx& ctx, const uint32_t* send, uint32_t* recv, size_t n) override {
    STB_NCCL(ctx, nccl().AllGather(send, recv, n, ncclUint32, comm, ctx.stream));
    return STB_OK;
  }
  uint32_t epoch = 0;  // every rank runs the same sequence of exchanges
  int exchange(Ctx& ctx, char* const* all, uint64_t recv_off, uint64_t flag_off, const uint32_t* send, uint32_t words, uint32_t send_stride,
               uint32_t* timeout_flag) override {
    PeerBox box{};
    for (int r = 0; r < world; ++r) box.base[r] = all[r];
    box.recv_off = recv_off;
    box.flag_off = flag_off;
    box.self = (uint32_t)rank;
    box.world = (uint32_t)world;
    peer_exchange_kernel<<<1, STB_MAX_RANKS * 32, 0, ctx.stream>>>(box, send, words, send_stride, ++epoch, timeout_flag);
    return STB_OK;
  }
  int share(Ctx& ctx, char* mine, char** all) override {
    epoch = 0;  // a new arena: its flags are zero
    cudaIpcMemHandle_t h;
    STB_CUDA(ctx, cudaIpcGetMemHandle(&h, mine));
    const size_t hb = sizeof(h);
    STB_CUDA(ctx, hbuf.ensure(hb * (size_t)(world + 1), ctx.stream));
    STB_CUDA(ctx, cudaMemcpyAsync(hbuf.ptr + hb * world, &h, hb, cudaMemcpyHostToDevice, ctx.stream));
    STB_NCCL(ctx, nccl().AllGather(hbuf.ptr + hb * world, hbuf.ptr, hb, ncclChar, comm, ctx.stream));
    std::vector<cudaIpcMemHandle_t> hs(world);
    STB_CUDA(ctx, cudaMemcpyAsync(hs.data(), hbuf.ptr, hb * world, cudaMemcpyDeviceToHost, ctx.stream));
    STB_CUDA(ctx, cudaStreamSynchronize(ctx.stream));
    for (int r = 0; r < world; ++r) {
      if (r == rank) {
        all[r] = mine;
        continue;
      }
      void* p = nullptr;
      STB_CUDA(ctx, cudaIpcOpenMemHandle(&p, hs[r], cudaIpcMemLazyEnablePeerAccess));
      all[r] = static_cast<char*>(p);
    }
    return STB_OK;
  }
  void unshare(char** all) override {
    for (int r = 0; r < world; ++r)
      if (r != rank && all[r]) cudaIpcCloseMemHandle(all[r]);
  }
  int gather_to_root(Ctx& ctx, const void* send, size_t bytes, void* recv, const size_t* bytes_of) override {
    STB_NCCL(ctx, nccl().GroupStart());
    if (rank == 0) {
      size_t off = 0;
      for (int r = 0; r < world; ++r) {
        if (r == 0) {
          if (bytes_of[0]) STB_CUDA(ctx, cudaMemcpyAsync(recv, send, bytes_of[0], cudaMemcpyDeviceToDevice, ctx.stream));
        } else if (bytes_of[r]) {
          STB_NCCL(ctx, nccl().Recv(static_cast<char*>(recv) + off, bytes_of[r], ncclChar, r, comm, ctx.stream));
        }
        off += bytes_of[r];
      }
    } else if (bytes) {
      STB_NCCL(ctx, nccl().Send(send, bytes, ncclChar, 0, comm, ctx.stream));
    }
    STB_NCCL(ctx, nccl().GroupEnd());
    return STB_OK;
  }
};

// Virtual ranks: threads of one process sharing one GPU (tests; a box with fewer GPUs than ranks).
// Every collective is a stream synchronisation plus a host barrier; no kernel ever waits for another.
struct LocalGroup {
  int world = 1;
  std::mutex m;
  std::condition_variable cv;
  int waiting = 0;
  uint64_t generation = 0;
  const void* slot[STB_MAX_RANKS] = {};
  size_t size[STB_MAX_RANKS] = {};
  void wait() {
    std::unique_lock<std::mutex> lk(m);
    const uint64_t gen = generation;
    if (++waiting == world) {
      waiting = 0;
      ++generation;
      cv.notify_all();
    } else {
      cv.wait(lk, [&] { return generation != gen; });
    }
  }
};

struct LocalComm : Comm {
  std::shared_ptr<LocalGroup> g;
  DevBuf<uint32_t> tmp;
  DevBuf<const uint32_t*> ptrs;
  int sync_all(Ctx& ctx) {
    STB_CUDA(ctx, cudaStreamSynchronize(ctx.stream));
    g->wait();
    return STB_OK;
  }
  int barrier(Ctx& ctx) override { return sync_all(ctx); }
  int all_reduce_min(Ctx& ctx, uint32_t* buf, size_t n) override {
    g->slot[rank] = buf;
    STB_TRY(sync_all(ctx));
    STB_CUDA(ctx, tmp.ensure(n, ctx.stream));
    STB_CUDA(ctx, ptrs.ensure(world, ctx.stream));
    std::vector<const uint32_t*> h(world);
    for (int r = 0; r < world; ++r) h[r] = static_cast<const uint32_t*>(g->slot[r]);
    STB_CUDA(ctx, cudaMemcpyAsync(ptrs.ptr, h.data(), world * sizeof(void*), cudaMemcpyHostToDevice, ctx.stream));
    min_over_ranks_kernel<<<592, 256, 0, ctx.stream>>>(tmp.ptr, ptrs.ptr, world, n);
    STB_TRY(sync_all(ctx));  // everybody has read everybody's input
    STB_CUDA(ctx, cudaMemcpyAsync(buf, tmp.ptr, n * 4, cudaMemcpyDeviceToDevice, ctx.stream));
    return STB_OK;
  }
  int all_gather_u32(Ctx& ctx, const uint32_t* send, uint32_t* recv, size_t n) override {
    g->slot[rank] = send;
    STB_TRY(sync_all(ctx));
    for (int r = 0; r < world; ++r) STB_CUDA(ctx, cudaMemcpyAsync(recv + (size_t)r * n, g->slot[r], n * 4, cudaMemcpyDeviceToDevice, ctx.stream));
    STB_TRY(sync_all(ctx));
    return STB_OK;
  }
  int exchange(Ctx& ctx, char* const* all, uint64_t recv_off, uint64_t, const uint32_t* send, uint32_t words, uint32_t send_stride, uint32_t*) override {
    // threads of one process: everybody's pointers are valid here; the host barrier orders the copies
    g->slot[rank] = send;
    STB_TRY(sync_all(ctx));
    for (int r = 0; r < world && words; ++r)
      STB_CUDA(ctx, cudaMemcpyAsync(all[rank] + recv_off + (uint64_t)r * XCHG_WORDS * 4, static_cast<const uint32_t*>(g->slot[r]) + (uint64_t)rank * send_stride,
                                    (size_t)words * 4, cudaMemcpyDeviceToDevice, ctx.stream));
    STB_TRY(sync_all(ctx));
    return STB_OK;
  }
  int share(Ctx& ctx, char* mine, char** all) override {
    g->slot[rank] = mine;
    STB_TRY(sync_all(ctx));
    for (int r = 0; r < world; ++r) all[r] = const_cast<char*>(static_cast<const char*>(g->slot[r]));
    STB_TRY(sync_all(ctx));
    return STB_OK;
  }
  void unshare(char**) override {}
  int gather_to_root(Ctx& ctx, const void* send, size_t bytes, void* recv, const size_t* bytes_of) override {
    g->slot[rank] = send;
    g->size[rank] = bytes;
    STB_TRY(sync_all(ctx));
    if (rank == 0) {
      size_t off = 0;
      for (int r = 0; r < world; ++r) {
        if (bytes_of[r]) STB_CUDA(ctx, cudaMemcpyAsync(static_cast<char*>(recv) + off, g->slot[r], bytes_of[r], cudaMemcpyDeviceToDevice, ctx.stream));
        off += bytes_of[r];
      }
    }
    STB_TRY(sync_all(ctx));
    return STB_OK;
  }
};

// ---- kernels of the sharded level loop -----------------------------------------------------------

// exclusive prefix of the tile counts (tilecnt, in place); one CTA per chunk of CHUNK_TILES tiles
__global__ void __launch_bounds__(LVL_THREADS) tile_prefix_kernel(uint32_t* __restrict__ tilecnt, const uint32_t* __restrict__ chunkcnt, uint32_t tiles) {
  __shared__ uint32_t warp_totals[LVL_THREADS / 32], chunks_before[LVL_THREADS / 32];
  const uint32_t t = blockIdx.x * CHUNK_TILES + threadIdx.x;
  uint32_t part = 0;
  for (uint32_t i = threadIdx.x; i < blockIdx.x; i += LVL_THREADS) part += chunkcnt[i];
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) chunks_before[threadIdx.x >> 5] = part;
  uint32_t before = block_exclusive_sum<LVL_THREADS>(t < tiles ? tilecnt[t] : 0u, warp_totals);  // its barrier publishes chunks_before
#pragma unroll
  for (int w = 0; w < LVL_THREADS / 32; ++w) before += chunks_before[w];
  if (t < tiles) tilecnt[t] = before;
}

// leaf ids: id(code) = rank of the code's first position; the leaf table in id order
__global__ void __launch_bounds__(256)
leaf_ids_kernel(const uint32_t* __restrict__ minpos, uint32_t entries, const uint32_t* __restrict__ bits, const uint32_t* __restrict__ tile_before,
                uint32_t* __restrict__ ids, unsigned long long* __restrict__ leaves, int S) {
  const uint32_t c = blockIdx.x * 256 + threadIdx.x;
  if (c >= entries) return;
  const uint32_t q = minpos[c];
  if (q == 0xffffffffu) return;
  const uint32_t tile = q / LVL_TILE, w0 = tile * (LVL_TILE / 32), w = q >> 5;
  uint32_t id = tile_before[tile] + __popc(bits[w] & ((1u << (q & 31)) - 1u));
  for (uint32_t i = w0; i < w; ++i) id += __popc(bits[i]);
  ids[c] = id;
  leaves[id] = leaf_from_2bit(c, S);
}

// The home rank applies the answers about its positions: it reads the list every owner kept for it
// (coalesced loads over NVLink; the lists' lengths arrived with the level's second exchange) and updates
// its own words.  answer = (flags | position) << 32 | first position (a later occurrence) or | 0xffffffff (a first
// occurrence whose key occurred again).  The lists are walked as one sequence, four loads in flight per thread:
// a peer's memory answers after a few microseconds.
__global__ void __launch_bounds__(256)
apply_answers_kernel(PeerHome home, uint32_t world, uint32_t* __restrict__ aux, uint32_t* __restrict__ first_bits, uint32_t* __restrict__ multi_bits) {
  __shared__ uint32_t before[STB_MAX_RANKS + 1];
  if (threadIdx.x == 0) {
    uint32_t sum = 0;
    for (uint32_t o = 0; o < world; ++o) {
      before[o] = sum;
      sum += min(__ldg(home.counts_in + o * home.counts_stride), home.ans_cap);
    }
    for (uint32_t o = world; o <= STB_MAX_RANKS; ++o) before[o] = sum;
  }
  __syncthreads();
  const uint32_t total = before[world], stride = gridDim.x * 256;
  const uint32_t mask = (1u << home.log2_positions) - 1u;
  for (uint32_t i0 = blockIdx.x * 256 + threadIdx.x; i0 < total; i0 += 4 * stride) {
    unsigned long long a[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t i = i0 + k * stride;
      a[k] = ~0ull;
      if (i < total) {
        uint32_t o = 0;
        while (before[o + 1] <= i) ++o;
        a[k] = __ldcs(reinterpret_cast<const unsigned long long*>(home.base[o] + home.ans_off) + (uint64_t)home.self * home.ans_cap + (i - before[o]));
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (a[k] == ~0ull) continue;
      const uint32_t pf = (uint32_t)(a[k] >> 32), p = pf & mask, fp = (uint32_t)a[k];
      if (fp == 0xffffffffu) {
        atomicOr(multi_bits + (p >> 5), 1u << (p & 31));
      } else {
        atomicAnd(first_bits + (p >> 5), ~(1u << (p & 31)));
        aux[p] = (pf & ~IDX_MASK) | fp;  // the node's flags came along in the record's position word
      }
    }
  }
}

// local number of first occurrences = sum of the chunk totals
__global__ void __launch_bounds__(256) sum_chunks_kernel(const uint32_t* __restrict__ chunkcnt, uint32_t chunks, uint32_t* __restrict__ out) {
  __shared__ uint32_t warp_totals[8];
  uint32_t s = 0;
  for (uint32_t i = threadIdx.x; i < chunks; i += 256) s += chunkcnt[i];
  uint32_t total;
  block_exclusive_sum<256>(s, warp_totals, &total);
  if (threadIdx.x == 0) *out = total;
}

// ids of this rank start after the first occurrences of the ranks before it
__global__ void id_base_kernel(const uint32_t* __restrict__ totals, uint32_t stride, int rank, int world, uint32_t* __restrict__ base,
                               uint32_t* __restrict__ level_total, uint32_t* __restrict__ keep) {
  uint32_t b = 0, t = 0;
  for (int r = 0; r < world; ++r) {
    const uint32_t v = totals[(uint64_t)r * stride];
    keep[r] = v;  // read by the host once, after the build
    if (r < rank) b += v;
    t += v;
  }
  *base = b;
  *level_total = t;
}

// later occurrences: the finished pointer of the first occurrence lives on its home rank
__global__ void __launch_bounds__(LVL_THREADS)
shard_resolve_kernel(const uint32_t* aux, uint32_t* __restrict__ out, uint32_t n, const uint32_t* bitmask, PeerHome home,
                     uint64_t ptr_off) {
  const uint32_t lane = threadIdx.x & 31;
#pragma unroll
  for (int it = 0; it < LVL_ITERS; ++it) {
    const uint32_t p = blockIdx.x * LVL_TILE + it * LVL_THREADS + threadIdx.x;
    if (p < n && !((bitmask[p >> 5] >> lane) & 1u)) {
      const uint32_t t = aux[p];
      uint32_t q = t & IDX_MASK;
      if ((q >> home.log2_positions) == home.self) {  // a run's head (bucket.cu) that is itself a later occurrence: one more hop
        const uint32_t ql = q & ((1u << home.log2_positions) - 1u);
        if (ql < p && p - ql < COLLAPSE_WINDOW && !((__ldcg(bitmask + (ql >> 5)) >> (ql & 31u)) & 1u)) q = __ldcg(aux + ql) & IDX_MASK;
      }
      const uint32_t* first = reinterpret_cast<const uint32_t*>(home.base[q >> home.log2_positions] + ptr_off) + (q & ((1u << home.log2_positions) - 1u));
      out[p] = finish_pointer(__ldcg(first) & IDX_MASK, t & ~IDX_MASK);
    }
  }
}

int log2_exact(uint64_t v) {
  int l = 0;
  while ((1ull << l) < v) ++l;
  return l;
}

}  // namespace

// ---- one rank of a sharded build ------------------------------------------------------------------
struct Shard : Ctx {
  Options opt;
  std::unique_ptr<Comm> comm;
  stb_tree* upper = nullptr;  // rank 0: the top of the tree (single-GPU code), then the gathered tree's source of truth

  // plan of the current build
  uint64_t n_leaves = 0, shard = 0, cut = 0;
  int pointer_levels = 0;  // sharded pointer levels (0 = leaf pointers); node layers 0 .. pointer_levels-2 are built sharded
  uint64_t level_total(int l) const { return ceil_div(n_leaves, 1ull << l); }
  void level_range(int r, int l, uint64_t* lo, uint64_t* hi) const {
    const uint64_t per = shard >> l, total = level_total(l);
    *lo = std::min<uint64_t>(total, (uint64_t)r * per);
    *hi = std::min<uint64_t>(total, (uint64_t)(r + 1) * per);
  }
  void plan(uint64_t n) {
    n_leaves = n;
    const int world = comm->world;
    const uint64_t per = std::max<uint64_t>(1, ceil_div(n, world));
    shard = 1;
    while (shard < per) shard <<= 1;
    // below this many positions a level costs less on rank 0 alone than its four exchanges and the pulls over
    // NVLink cost the world (measured at 3.1 Gbp: 8 M / 4 M / 2-4 M positions at 2 / 4 / 8 ranks, profiles/README.md)
    cut = opt_cut ? opt_cut : std::max<uint64_t>(1ull << 20, (1ull << 24) / world);
    pointer_levels = 1;
    while ((shard >> pointer_levels) >= 1 && level_total(pointer_levels) > cut && level_total(pointer_levels) > 1) ++pointer_levels;
  }
  uint64_t opt_cut = 0;

  // peer-visible arena (cudaMalloc: CUDA IPC cannot export pool memory)
  char* arena = nullptr;
  uint64_t arena_bytes = 0, arena_shard = 0;
  char* peers[STB_MAX_RANKS] = {};
  bool shared = false;
  uint64_t off_ptr[2] = {}, off_aux = 0, off_first[2] = {}, off_multi[2] = {}, off_seg_keys = 0, off_seg_pos = 0, off_seg_count = 0;
  uint64_t off_ans = 0, off_ans_count = 0, ans_records = 0;
  uint64_t off_box = 0, off_flags = 0;  // mailboxes and epoch flags of Comm::exchange
  uint64_t box_off(int slot) const { return off_box + (uint64_t)slot * STB_MAX_RANKS * XCHG_WORDS * 4; }
  const uint32_t* box(int slot) const { return reinterpret_cast<const uint32_t*>(arena + box_off(slot)); }
  int exchange(int slot, const uint32_t* send, uint32_t words, uint32_t stride) {
    return comm->exchange(*this, peers, box_off(slot), off_flags, send, words, stride, scalars.ptr + 6);
  }

  // local scratch and results
  DevBuf<uint32_t> dminpos, dids, leaf_bits, tilecnt, count2, scalars, totals_all;
  BucketWorkspace ws;
  DevBuf<char> staging;                // host input lands here
  DevBuf<unsigned long long> leaves;   // the whole leaf table (every rank computes it; rank 0's is the tree's)
  std::vector<DevBuf<uint2>> slices;   // this rank's id range of every sharded node layer
  std::vector<uint32_t> h_totals;      // [level][rank] unique counts (level 0 = leaves: [0] only), after a build
  uint32_t h_leaves = 0;
  bool built = false;
  bool whole_on_root = false;  // the last build fell back to rank 0 alone (skewed keys): `upper` holds the whole tree
  uint64_t builds = 0;

  ~Shard() {
    if (shared) comm->unshare(peers);
    if (arena) cudaFree(arena);
  }
};

namespace {

int ensure_arena(Shard& s) {
  // sized by the shard (leaf positions per rank): every level fits in what the first ones need
  if (s.arena && s.arena_shard >= s.shard) return STB_OK;
  if (s.shared) {
    STB_TRY(s.comm->barrier(s));
    STB_CUDA(s, cudaStreamSynchronize(s.stream));
    s.comm->unshare(s.peers);
    s.shared = false;
  }
  if (s.arena) STB_CUDA(s, cudaFree(s.arena));
  s.arena = nullptr;
  const uint64_t P = std::max<uint64_t>(s.shard / 2, 1);  // node positions per rank at the first node level
  uint64_t off = 0;
  auto carve = [&](uint64_t bytes) {
    const uint64_t at = off;
    off += (bytes + 255) & ~255ull;
    return at;
  };
  s.off_ptr[0] = carve(s.shard * 4);
  s.off_ptr[1] = carve(P * 4);
  s.off_aux = carve(P * 4);
  for (int i = 0; i < 2; ++i) {
    s.off_first[i] = carve(ceil_div(P, LVL_TILE) * (LVL_TILE / 8));
    s.off_multi[i] = carve(ceil_div(P, LVL_TILE) * (LVL_TILE / 8));
  }
  // this rank's first-pass buckets at the largest level (mean P / 2^b1 records each, with head-room; at most
  // 2^9 buckets), and the answers it keeps for every home rank
  const uint64_t seg_records = P + P * s.opt.bucket_slack_permille / 1000 + 512ull * 512;
  s.off_seg_keys = carve(seg_records * 8);
  s.off_seg_pos = carve(seg_records * 4);
  s.off_seg_count = carve(512ull * 4);
  s.ans_records = 2 * P / (uint64_t)s.comm->world + 65536;  // per home rank
  s.off_ans = carve(s.ans_records * 8 * (uint64_t)s.comm->world);
  s.off_ans_count = carve(STB_MAX_RANKS * 4);
  s.off_box = carve((uint64_t)XCHG_SLOTS * STB_MAX_RANKS * XCHG_WORDS * 4);
  s.off_flags = carve(STB_MAX_RANKS * 4);
  s.arena_bytes = off;
  STB_CUDA(s, cudaMalloc(&s.arena, s.arena_bytes));
  STB_CUDA(s, cudaMemsetAsync(s.arena + s.off_flags, 0, STB_MAX_RANKS * 4, s.stream));  // before anybody can see the arena
  s.arena_shard = s.shard;
  STB_TRY(s.comm->share(s, s.arena, s.peers));
  s.shared = true;
  return STB_OK;
}

// Bucket shape of a sharded level of n positions in total, P per rank.
ShardBuckets level_buckets(const Shard& s, uint64_t n_total, uint64_t P, int level_parity, int out_ptr) {
  ShardBuckets sb;
  const int lw = log2_exact(s.comm->world);
  sb.cap2 = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(s.opt.bucket_cap, 16), 3072);
  int bits = 2;
  while (bits < 18 && (n_total >> bits) > (uint64_t)sb.cap2 * 2 / 3) ++bits;
  bits = std::max(bits, lw + 2);
  sb.b1 = std::max((bits + 1) / 2, lw + 1);
  sb.b1 = std::min(sb.b1, 9);
  sb.b2 = std::max(1, std::min(bits - sb.b1, 9));
  const uint64_t mean = ceil_div(P, 1ull << sb.b1);
  sb.cap_seg = (uint32_t)((mean + mean * s.opt.bucket_slack_permille / 1000 + 256 + 3) & ~3ull);
  sb.dest.bucket_shift = (uint32_t)(sb.b1 - lw);
  sb.dest.src = (uint32_t)s.comm->rank;
  sb.dest.world = (uint32_t)s.comm->world;
  sb.dest.keys_off = s.off_seg_keys;
  sb.dest.pos_off = s.off_seg_pos;
  sb.dest.count_off = s.off_seg_count;
  sb.home.ans_off = s.off_ans;
  sb.home.ans_count_off = s.off_ans_count;
  sb.home.ans_cap = (uint32_t)std::min<uint64_t>(s.ans_records, 0xffffffffull);
  sb.home.self = (uint32_t)s.comm->rank;
  sb.home.log2_positions = (uint32_t)log2_exact(P);
  for (int r = 0; r < s.comm->world; ++r) sb.dest.base[r] = sb.home.base[r] = s.peers[r];
  sb.dest.counts_in = s.box(0);
  sb.dest.counts_stride = XCHG_WORDS;
  sb.home.counts_in = s.box(1);
  sb.home.counts_stride = XCHG_WORDS;
  (void)level_parity;
  (void)out_ptr;
  return sb;
}

int shard_build(Shard& s, const char* d_body, uint64_t n_bases_total) {
  const int S = s.S;
  Comm& comm = *s.comm;
  const int rank = comm.rank, world = comm.world;
  cudaStream_t st = s.stream;
  if (S > 12) return s.fail(STB_ERR_INVALID_ARG, "sharded build: dna_size > 12 is not supported (use the single-GPU build)");
  const uint64_t n0 = n_bases_total / (uint64_t)S;
  if (n0 == 0) return s.fail(STB_ERR_EMPTY, "input holds fewer than dna_size bases");
  if (n0 >= (1ull << 30)) return s.fail(STB_ERR_TOO_LARGE, "2^30 or more leaf positions");
  s.built = false;
  s.plan(n0);
  STB_TRY(ensure_arena(s));
  uint64_t lo0, hi0;
  s.level_range(rank, 0, &lo0, &hi0);
  const uint64_t n_local = hi0 - lo0;
  const int L = s.pointer_levels;

  s.profile_level = s.opt.profile_levels ? 0 : -1;
  // ---- leaf level: replicated direct table, all-reduce(min) of the first positions, ids everywhere ----
  const uint64_t entries = 1ull << (2 * S);
  const uint64_t canon_entries = std::max<uint64_t>(entries / 2, 1);  // a canonical code's first nucleotide is A or C (dna.cpp:135-143)
  STB_CUDA(s, s.dminpos.ensure(entries, st));
  STB_CUDA(s, s.dids.ensure(entries, st));
  STB_CUDA(s, s.leaf_bits.ensure(ceil_div(n0, LVL_TILE) * (LVL_TILE / 32), st));
  {
    const uint64_t tiles = ceil_div(n0, LVL_TILE);
    STB_CUDA(s, s.tilecnt.ensure(tiles + tiles / CHUNK_TILES + 2, st));
  }
  STB_CUDA(s, s.scalars.ensure(8, st));  // [0] local total, [1] id base, [2] level total, [3] overflow, [4] leaf flag, [5] assign's total, [6] barrier timeout
  STB_CUDA(s, s.totals_all.ensure((uint64_t)world * 48 + 48, st));
  STB_CUDA(s, s.leaves.ensure(std::min<uint64_t>(n0, canon_entries) + 1, st));
  STB_CUDA(s, cudaMemsetAsync(s.scalars.ptr, 0, 8 * 4, st));
  STB_CUDA(s, cudaMemsetAsync(s.totals_all.ptr, 0, ((uint64_t)world * 48 + 48) * 4, st));
  STB_CUDA(s, cudaMemsetAsync(s.dminpos.ptr, 0xff, entries * 4, st));
  uint32_t* ptr_cur = reinterpret_cast<uint32_t*>(s.arena + s.off_ptr[0]);
  uint32_t* ptr_nxt = reinterpret_cast<uint32_t*>(s.arena + s.off_ptr[1]);
  int cur_which = 0;
  {
    int non_acgt = 0;
    const int rc = dist_leaf_direct_minpos(s, d_body, n_local, lo0, s.dminpos.ptr, ptr_cur, &non_acgt);
    if (rc != STB_OK && rc != STB_ERR_UNKNOWN_SYMBOL) return rc;
    // every rank must take the same path: an unknown symbol, or one outside ACGT, anywhere stops the
    // sharded build everywhere (the collectives below would otherwise wait for the rank that left)
    uint32_t flag = rc != STB_OK ? 2u : (non_acgt ? 1u : 0u);
    STB_CUDA(s, cudaMemcpyAsync(s.scalars.ptr + 4, &flag, 4, cudaMemcpyHostToDevice, st));
    STB_TRY(comm.all_gather_u32(s, s.scalars.ptr + 4, s.totals_all.ptr, 1));
    std::vector<uint32_t> flags(world);
    STB_CUDA(s, cudaMemcpyAsync(flags.data(), s.totals_all.ptr, world * 4, cudaMemcpyDeviceToHost, st));
    STB_CUDA(s, cudaStreamSynchronize(st));
    if (rc != STB_OK) return rc;  // this rank's own message (src/dna.cpp:44-47)
    for (uint32_t f : flags) {
      if (f == 2u) return s.fail(STB_ERR_UNKNOWN_SYMBOL, "Encountered unknown symbol (in another rank's part of the text)");
      if (f == 1u) return s.fail(STB_ERR_INVALID_ARG, "sharded build: the text holds symbols other than ACGT (use the single-GPU build)");
    }
    STB_CUDA(s, cudaMemsetAsync(s.totals_all.ptr, 0, world * 4, st));
  }
  {
    Launch l(s, "collective_leaf_min", false);
    STB_TRY(comm.all_reduce_min(s, s.dminpos.ptr, canon_entries));
  }
  {
    const uint32_t tiles = (uint32_t)ceil_div(n0, LVL_TILE), chunks = tiles / CHUNK_TILES + 1;
    uint32_t* chunkcnt = s.tilecnt.ptr + tiles;
    STB_CUDA(s, cudaMemsetAsync(s.leaf_bits.ptr, 0, (uint64_t)tiles * (LVL_TILE / 8), st));
    STB_CUDA(s, cudaMemsetAsync(chunkcnt, 0, (uint64_t)chunks * 4, st));
    Launch l(s, "shard_leaf_ids");
    mark_first_kernel<<<(unsigned)ceil_div(canon_entries, 256), 256, 0, st>>>(s.dminpos.ptr, (uint32_t)canon_entries, s.leaf_bits.ptr);
    count_kernel<<<(unsigned)ceil_div((uint64_t)tiles * 32, 256), 256, 0, st>>>(s.leaf_bits.ptr, 0u, tiles, s.tilecnt.ptr, chunkcnt);
    sum_chunks_kernel<<<1, 256, 0, st>>>(chunkcnt, chunks, s.totals_all.ptr);  // level 0 total: the same on every rank
    tile_prefix_kernel<<<chunks, LVL_THREADS, 0, st>>>(s.tilecnt.ptr, chunkcnt, tiles);
    leaf_ids_kernel<<<(unsigned)ceil_div(canon_entries, 256), 256, 0, st>>>(s.dminpos.ptr, (uint32_t)canon_entries, s.leaf_bits.ptr, s.tilecnt.ptr, s.dids.ptr,
                                                                           s.leaves.ptr, S);
  }
  // with at least one sharded node level, its partition pass finishes the leaf words on the way (bucket.cuh: LeafFinish)
  const bool fuse_leaf = L > 1;
  if (n_local && !fuse_leaf) {
    Launch l(s, "shard_leaf_pointers");
    finish_leaves_kernel<<<(unsigned)ceil_div(n_local, 256), 256, 0, st>>>(ptr_cur, n_local, s.dids.ptr, ptr_cur);
  }

  // ---- sharded node levels ----
  s.slices.clear();
  uint64_t n_cur_local = n_local;
  for (int j = 0; j + 1 < L; ++j) {  // node layer j: pointer level j -> pointer level j + 1
    uint64_t lo, hi;
    s.level_range(rank, j + 1, &lo, &hi);
    const uint64_t n_next_local = hi - lo, P = s.shard >> (j + 1), n_total = s.level_total(j + 1);
    const int par = j & 1;
    if (s.opt.profile_levels) s.profile_level = j + 1;
    uint32_t* first_bits = reinterpret_cast<uint32_t*>(s.arena + s.off_first[par]);
    uint32_t* multi_bits = reinterpret_cast<uint32_t*>(s.arena + s.off_multi[par]);
    uint32_t* aux = reinterpret_cast<uint32_t*>(s.arena + s.off_aux);
    const uint32_t* child_first = (j > 0 && s.opt.child_filter) ? reinterpret_cast<uint32_t*>(s.arena + s.off_first[par ^ 1]) : nullptr;
    const uint32_t* child_multi = (j > 0 && s.opt.child_filter) ? reinterpret_cast<uint32_t*>(s.arena + s.off_multi[par ^ 1]) : nullptr;
    const ShardBuckets sb = level_buckets(s, n_total, P, par, cur_which ^ 1);
    const uint32_t nb1 = 1u << sb.b1, local1 = 1u << sb.dest.bucket_shift;
    if ((uint64_t)nb1 * sb.cap_seg > (s.off_seg_pos - s.off_seg_keys) / 8)
      return s.fail(STB_ERR_TOO_LARGE, "sharded build: bucket arena too small for this level (raise bucket_slack_permille)");
    const uint64_t words = ceil_div(std::max<uint64_t>(P, 1), LVL_TILE) * (LVL_TILE / 32);
    unsigned long long* seg_keys = reinterpret_cast<unsigned long long*>(s.arena + s.off_seg_keys);
    uint32_t* seg_pos = reinterpret_cast<uint32_t*>(s.arena + s.off_seg_pos);
    uint32_t* seg_count = reinterpret_cast<uint32_t*>(s.arena + s.off_seg_count);
    STB_CUDA(s, cudaMemsetAsync(first_bits, 0, words * 4, st));
    STB_CUDA(s, cudaMemsetAsync(multi_bits, 0, words * 4, st));
    STB_CUDA(s, cudaMemsetAsync(seg_count, 0, 512 * 4, st));
    STB_CUDA(s, cudaMemsetAsync(s.arena + s.off_ans_count, 0, STB_MAX_RANKS * 4, st));
    const LeafFinish leaf_finish{ptr_cur, nullptr, s.dids.ptr, nullptr};
    STB_TRY(shard_partition(s, sb, ptr_cur, (uint32_t)n_cur_local, (uint32_t)n_next_local, (uint32_t)lo, child_first, child_multi, aux, first_bits,
                            multi_bits, seg_keys, seg_pos, seg_count, s.scalars.ptr + 3, (j == 0 && fuse_leaf) ? &leaf_finish : nullptr));
    {
      Launch l(s, "peer_exchange");
      STB_TRY(s.exchange(0, seg_count, local1, local1));  // every rank's buckets are complete and the owners know their sizes: they pull them
    }
    STB_CUDA(s, s.count2.ensure((uint64_t)local1 << sb.b2, st));
    STB_TRY(shard_dedup(s, sb, s.ws, s.count2.ptr, s.scalars.ptr + 3));
    {
      Launch l(s, "peer_exchange");
      STB_TRY(s.exchange(1, reinterpret_cast<const uint32_t*>(s.arena + s.off_ans_count), 1, 1));  // the answer lists are complete, their lengths delivered
    }
    if (s.opt.profile_levels > 1) {  // debugging aid: how many answers this owner keeps for every home rank
      uint32_t kept[STB_MAX_RANKS];
      STB_CUDA(s, cudaMemcpyAsync(kept, s.arena + s.off_ans_count, sizeof(kept), cudaMemcpyDeviceToHost, st));
      STB_CUDA(s, cudaStreamSynchronize(st));
      std::string line = "[stb shard " + std::to_string(rank) + "/" + std::to_string(world) + " node layer " + std::to_string(j) + "] answers kept per home rank:";
      for (int r = 0; r < world; ++r) line += " " + std::to_string(kept[r]);
      fprintf(stderr, "%s\n", line.c_str());
    }
    {
      Launch l(s, "shard_apply");
      apply_answers_kernel<<<1184, 256, 0, st>>>(sb.home, (uint32_t)world, aux, first_bits, multi_bits);
    }
    // ids: local counts -> the world's totals -> this rank's base
    const uint32_t tiles = (uint32_t)ceil_div(n_next_local, LVL_TILE), chunks = tiles / CHUNK_TILES + 1;
    uint32_t* chunkcnt = s.tilecnt.ptr + tiles;
    STB_CUDA(s, cudaMemsetAsync(chunkcnt, 0, (uint64_t)chunks * 4, st));
    if (tiles) {
      Launch l(s, "count_firsts");
      count_kernel<<<(unsigned)ceil_div((uint64_t)tiles * 32, 256), 256, 0, st>>>(first_bits, 0u, tiles, s.tilecnt.ptr, chunkcnt);
    }
    sum_chunks_kernel<<<1, 256, 0, st>>>(chunkcnt, chunks, s.scalars.ptr);
    uint32_t* totals = s.totals_all.ptr + (uint64_t)(j + 1) * world;
    {
      Launch l(s, "peer_exchange");
      STB_TRY(s.exchange(2, s.scalars.ptr, 1, 0));  // everybody's number of first occurrences
    }
    id_base_kernel<<<1, 1, 0, st>>>(s.box(2), XCHG_WORDS, rank, world, s.scalars.ptr + 1, s.scalars.ptr + 2, totals);
    s.slices.emplace_back();
    STB_CUDA(s, s.slices.back().alloc(std::max<uint64_t>(n_next_local, 1), st));
    if (tiles) {
      Launch l(s, "assign_ids");
      LevelTable none{nullptr, nullptr, nullptr, 0u};
      assign_kernel<MODE_NODE><<<tiles, LVL_THREADS, 0, st>>>(ptr_nxt, (uint32_t)n_next_local, none, first_bits, s.tilecnt.ptr, chunkcnt, 0u, nullptr,
                                                              s.scalars.ptr + 5, s.slices.back().ptr, S, ptr_cur, (uint32_t)n_cur_local, s.scalars.ptr + 1);
    }
    {
      Launch l(s, "peer_exchange");
      STB_TRY(s.exchange(3, nullptr, 0, 0));  // every rank's first occurrences have their ids
    }
    if (tiles) {
      Launch l(s, "shard_resolve");
      shard_resolve_kernel<<<tiles, LVL_THREADS, 0, st>>>(aux, ptr_nxt, (uint32_t)n_next_local, first_bits, sb.home, s.off_ptr[cur_which ^ 1]);
    }
    std::swap(ptr_cur, ptr_nxt);
    cur_which ^= 1;
    n_cur_local = n_next_local;
  }

  // ---- the top of the tree on rank 0 ----
  s.profile_level = s.opt.profile_levels ? L : -1;
  STB_TRY(s.exchange(0, nullptr, 0, 0));  // every rank's last pointer array is final
  const uint64_t n_top = s.level_total(L - 1);
  if (rank == 0) {
    Launch l(s, "root_top_levels", false);
    DevBuf<uint32_t> top;
    STB_CUDA(s, top.alloc(n_top, st));
    for (int r = 0; r < world; ++r) {
      uint64_t lo, hi;
      s.level_range(r, L - 1, &lo, &hi);
      if (hi > lo)
        STB_CUDA(s, cudaMemcpyAsync(top.ptr + lo, s.peers[r] + s.off_ptr[cur_which], (hi - lo) * 4, cudaMemcpyDeviceToDevice, st));
    }
    Tree& up = *s.upper;
    up.opt = s.opt;
    up.stream = st;
    const int rc = build_upper_levels(up, top.ptr, n_top, L == 1);
    if (rc != STB_OK) return s.fail(rc, up.error);
  }
  STB_TRY(s.exchange(1, nullptr, 0, 0));  // rank 0 has read the peers' arrays: the arenas may be reused

  s.profile_level = -1;
  // ---- what the host needs to know, once ----
  s.h_totals.assign((size_t)L * world, 0);
  std::vector<uint32_t> overflowed(world);
  uint32_t* gathered_flags = s.totals_all.ptr + (uint64_t)world * 47;
  STB_TRY(comm.all_gather_u32(s, s.scalars.ptr + 3, gathered_flags, 1));
  STB_CUDA(s, cudaMemcpyAsync(s.h_totals.data(), s.totals_all.ptr, s.h_totals.size() * 4, cudaMemcpyDeviceToHost, st));
  STB_CUDA(s, cudaMemcpyAsync(overflowed.data(), gathered_flags, world * 4, cudaMemcpyDeviceToHost, st));
  uint32_t timed_out = 0;
  STB_CUDA(s, cudaMemcpyAsync(&timed_out, s.scalars.ptr + 6, 4, cudaMemcpyDeviceToHost, st));
  STB_CUDA(s, cudaStreamSynchronize(st));
  STB_CUDA(s, cudaGetLastError());
  if (timed_out) return s.fail(STB_ERR_CUDA, "sharded build: a rank did not reach a level's barrier within half a minute (did it fail on its own?)");
  s.whole_on_root = false;
  for (uint32_t f : overflowed)
    if (f) s.whole_on_root = true;
  if (s.whole_on_root) {
    // A bucket overflowed somewhere: the keys are too skewed for fixed-size buckets (a handful of
    // distinct keys, as with dna_size 1).  Every rank knows; the text goes to rank 0, which builds the
    // whole tree with the single-GPU code (that has the hash-table path for such levels).
    std::vector<size_t> bytes(world);
    for (int r = 0; r < world; ++r) {
      uint64_t lo, hi;
      s.level_range(r, 0, &lo, &hi);
      bytes[r] = (size_t)(hi - lo) * S;
    }
    DevBuf<char> whole;
    if (rank == 0) STB_CUDA(s, whole.alloc(n0 * (uint64_t)S + 16, st));
    STB_TRY(comm.gather_to_root(s, d_body, bytes[rank], whole.ptr, bytes.data()));
    if (rank == 0) {
      Tree& up = *s.upper;
      up.opt = s.opt;
      up.stream = st;
      const int rc = build_from_body(up, whole.ptr, n0 * (uint64_t)S);
      if (rc != STB_OK) return s.fail(rc, up.error);
      s.h_totals.assign((size_t)L * world, 0);
      s.h_totals[0] = (uint32_t)up.n_leaves;
    }
    STB_CUDA(s, cudaStreamSynchronize(st));
    s.pointer_levels = 1;
  }
  s.h_leaves = s.h_totals[0];
  s.built = true;
  ++s.builds;
  return STB_OK;
}

}  // namespace

}  // namespace stb

using namespace stb;

struct stb_shard : stb::Shard {};

extern "C" {

int stb_shard_unique_id(uint8_t id[STB_SHARD_ID_BYTES]) {
  if (!id) return STB_ERR_INVALID_ARG;
  static_assert(STB_SHARD_ID_BYTES == NCCL_UNIQUE_ID_BYTES, "id size");
  if (!nccl().ok) return STB_ERR_CUDA;
  ncclUniqueId u;
  if (nccl().GetUniqueId(&u) != ncclSuccess) return STB_ERR_CUDA;
  memcpy(id, u.internal, STB_SHARD_ID_BYTES);
  return STB_OK;
}

static int shard_new(stb_shard** out, int device, int dna_size, void* cuda_stream) {
  if (!out) return STB_ERR_INVALID_ARG;
  *out = nullptr;
  if (dna_size < 1 || dna_size > 16) return STB_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return STB_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return STB_ERR_CUDA;
  stb_shard* s = new (std::nothrow) stb_shard();
  if (!s) return STB_ERR_INVALID_ARG;
  s->device = device;
  s->S = dna_size;
  s->stream = (cudaStream_t)cuda_stream;
  *out = s;
  return STB_OK;
}

int stb_shard_create(stb_shard** out, int device, int dna_size, void* cuda_stream, int rank, int world, const uint8_t id[STB_SHARD_ID_BYTES]) {
  if (!id || world < 1 || world > STB_MAX_RANKS || (world & (world - 1)) || rank < 0 || rank >= world) return STB_ERR_INVALID_ARG;
  if (!nccl().ok) return STB_ERR_CUDA;
  STB_TRY(shard_new(out, device, dna_size, cuda_stream));
  stb_shard* s = *out;
  auto* c = new NcclComm();
  c->rank = rank;
  c->world = world;
  s->comm.reset(c);
  ncclUniqueId u;
  memcpy(u.internal, id, STB_SHARD_ID_BYTES);
  if (nccl().CommInitRank(&c->comm, world, u, rank) != ncclSuccess) {
    delete s;
    *out = nullptr;
    return STB_ERR_CUDA;
  }
  if (rank == 0 && stb_create(&s->upper, device, dna_size, cuda_stream) != STB_OK) {
    delete s;
    *out = nullptr;
    return STB_ERR_CUDA;
  }
  return STB_OK;
}

int stb_shard_create_local(stb_shard** out, int world, int device, int dna_size) {
  if (!out || world < 1 || world > STB_MAX_RANKS || (world & (world - 1))) return STB_ERR_INVALID_ARG;
  auto group = std::make_shared<LocalGroup>();
  group->world = world;
  for (int r = 0; r < world; ++r) {
    cudaStream_t st = nullptr;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) return STB_ERR_CUDA;
    STB_TRY(shard_new(&out[r], device, dna_size, st));
    auto* c = new LocalComm();
    c->rank = r;
    c->world = world;
    c->g = group;
    out[r]->comm.reset(c);
    if (r == 0 && stb_create(&out[r]->upper, device, dna_size, st) != STB_OK) return STB_ERR_CUDA;
  }
  return STB_OK;
}

int stb_shard_destroy(stb_shard* s) {
  if (!s) return STB_OK;
  cudaSetDevice(s->device);
  cudaStreamSynchronize(s->stream);
  if (s->upper) stb_destroy(s->upper);
  delete s;
  return STB_OK;
}

int stb_shard_set_option(stb_shard* s, const char* name, uint64_t value) {
  if (!s || !name) return STB_ERR_INVALID_ARG;
  if (strcmp(name, "cut") == 0) {
    s->opt_cut = value;
    return STB_OK;
  }
  stb_tree tmp;
  tmp.opt = s->opt;
  const int rc = stb_set_option(&tmp, name, value);
  if (rc == STB_OK) s->opt = tmp.opt;
  return rc;
}

int stb_shard_range(const stb_shard* s, uint64_t n_bases_total, uint64_t* first_base, uint64_t* base_count) {
  if (!s || !first_base || !base_count) return STB_ERR_INVALID_ARG;
  stb_shard& m = const_cast<stb_shard&>(*s);
  const uint64_t keep = m.n_leaves;
  m.plan(n_bases_total / (uint64_t)s->S);
  uint64_t lo, hi;
  m.level_range(s->comm->rank, 0, &lo, &hi);
  *first_base = lo * (uint64_t)s->S;
  *base_count = (hi - lo) * (uint64_t)s->S;
  if (keep) m.plan(keep);
  return STB_OK;
}

int stb_shard_build_from_body(stb_shard* s, const char* body_local, uint64_t n_bases_total, int memory) {
  if (!s || (memory != STB_HOST && memory != STB_DEVICE)) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(s->device) != cudaSuccess) return STB_ERR_CUDA;
  uint64_t first = 0, count = 0;
  STB_TRY(stb_shard_range(s, n_bases_total, &first, &count));
  const char* d = body_local;
  if (memory == STB_HOST || (reinterpret_cast<uintptr_t>(body_local) & 15u)) {
    // the handle's grow-only staging buffer: no device allocation per call in steady state
    STB_CUDA(*s, s->staging.ensure(count + 16, s->stream));
    if (count)
      STB_CUDA(*s, cudaMemcpyAsync(s->staging.ptr, body_local, count, memory == STB_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, s->stream));
    d = s->staging.ptr;
  }
  return shard_build(*s, d, n_bases_total);
}

int stb_shard_layer_totals(const stb_shard* s, uint64_t* out, uint64_t cap, uint64_t* count) {
  if (!s || !count) return STB_ERR_INVALID_ARG;
  if (!s->built) return s->fail(STB_ERR_NOT_BUILT, "no sharded build yet");
  const int world = s->comm->world, L = s->pointer_levels;
  *count = (uint64_t)L;
  for (int l = 0; l < L && out && (uint64_t)l < cap; ++l) {
    uint64_t t = 0;
    if (l == 0) t = s->h_totals[0];
    else
      for (int r = 0; r < world; ++r) t += s->h_totals[(size_t)l * world + r];
    out[l] = t;
  }
  return STB_OK;
}

int stb_shard_gather(stb_shard* s, stb_tree* out) {
  if (!s || (s->comm->rank == 0 && !out)) return STB_ERR_INVALID_ARG;
  if (!s->built) return s->fail(STB_ERR_NOT_BUILT, "no sharded build yet");
  if (cudaSetDevice(s->device) != cudaSuccess) return STB_ERR_CUDA;
  Comm& comm = *s->comm;
  const int world = comm.world, rank = comm.rank, L = s->pointer_levels;
  cudaStream_t st = s->stream;
  Tree* t = rank == 0 ? out : nullptr;
  if (t) {
    t->clear();
    t->stream = st;
    const unsigned long long* leaf_table = s->whole_on_root ? s->upper->leaves.ptr : s->leaves.ptr;
    STB_CUDA(*s, t->leaves.alloc(s->h_leaves, st));
    STB_CUDA(*s, cudaMemcpyAsync(t->leaves.ptr, leaf_table, (uint64_t)s->h_leaves * 8, cudaMemcpyDeviceToDevice, st));
  }
  for (int j = 0; j + 1 < L; ++j) {
    std::vector<size_t> bytes(world);
    uint64_t total = 0;
    for (int r = 0; r < world; ++r) {
      bytes[r] = (size_t)s->h_totals[(size_t)(j + 1) * world + r] * sizeof(uint2);
      total += s->h_totals[(size_t)(j + 1) * world + r];
    }
    void* dst = nullptr;
    if (t) {
      t->layers.emplace_back();
      t->layers.back().count = total;
      STB_CUDA(*s, t->layers.back().nodes.alloc(total, st));
      dst = t->layers.back().nodes.ptr;
    }
    STB_TRY(comm.gather_to_root(*s, s->slices[j].ptr, bytes[rank], dst, bytes.data()));
  }
  if (t) {
    Tree& up = *s->upper;
    for (auto& layer : up.layers) {
      t->layers.emplace_back();
      t->layers.back().count = layer.count;
      STB_CUDA(*s, t->layers.back().nodes.alloc(layer.count, st));
      STB_CUDA(*s, cudaMemcpyAsync(t->layers.back().nodes.ptr, layer.nodes.ptr, layer.count * sizeof(uint2), cudaMemcpyDeviceToDevice, st));
    }
    t->n_leaves = s->h_leaves;
    t->root = up.root;
    t->width = s->n_leaves;
    t->built = true;
    t->plan_valid = false;
  }
  STB_CUDA(*s, cudaStreamSynchronize(st));
  return STB_OK;
}

const char* stb_shard_last_error(const stb_shard* s) { return s ? s->error.c_str() : "null handle"; }

int stb_shard_profile(stb_shard* s, int on, const char** names, double* total_ms, uint64_t* launches, uint64_t cap, uint64_t* count) {
  if (!s) return STB_ERR_INVALID_ARG;
  if (cudaSetDevice(s->device) != cudaSuccess) return STB_ERR_CUDA;
  s->flush_profile();
  if (count) {
    uint64_t i = 0;
    for (const auto& name : s->acc_order) {
      if (i < cap && names && total_ms && launches) {
        const auto& a = s->acc.at(name);
        names[i] = s->acc.find(name)->first.c_str();
        total_ms[i] = a.ms;
        launches[i] = a.launches;
      }
      ++i;
    }
    *count = i;
  }
  if (on < 0) {  // reset
    s->acc.clear();
    s->acc_order.clear();
  } else {
    s->profiling = on != 0;
  }
  return STB_OK;
}

}  // extern "C"
