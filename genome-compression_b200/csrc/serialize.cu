// serialize.cu — the .dag byte stream (reference src/shared_tree.cpp:488-546).
//
// Layout (all integers big-endian, include/utility.h:178-184):
//   pointer root | u64 leaf_count | leaf_count x ceil(S/2) bytes |
//   per node layer bottom-up: u64 node_count | node_count x (pointer left, pointer right)
// pointer = 1..4 bytes: segment(2) transpose(1) mirror(1) offset-high(4), then the
// remaining offset bytes (src/shared_tree.cpp:25-67, :122-142).
//
// The reference writes one byte at a time through ostream::put.  Here a plan pass
// sums the encoded length of every 1024-node tile, a scan turns the sums into byte
// offsets, and the emit pass has each CTA encode its tile into shared memory and
// store it as aligned words.  bytes() is the plan's grand total.
#include <algorithm>
#include <cstring>

#include "scan.cuh"
#include "staging.cuh"
#include "tree.h"

namespace stb {

constexpr int SER_THREADS = 256;
constexpr int SER_PER_THREAD = 4;
constexpr int SER_TILE = SER_THREADS * SER_PER_THREAD;  // 1024 nodes or leaves per CTA

// encoded length of a pointer: 1 + segment (src/shared_tree.cpp:44-49, :122-125)
__host__ __device__ __forceinline__ uint32_t ptr_len(uint32_t raw) {
  const uint32_t idx = raw & IDX_MASK;
  return 1u + (idx >= 16u) + (idx >= 4112u) + (idx >= 1052688u);
}

// writes the 1..4 bytes of a pointer; returns the length
__host__ __device__ __forceinline__ uint32_t ptr_encode(uint32_t raw, uint8_t* out) {
  const uint32_t idx = raw & IDX_MASK;
  uint32_t seg, off;
  if (idx == IDX_MASK) { seg = 3; off = 0xfffffffu; }
  else if (idx < 16u) { seg = 0; off = idx; }
  else if (idx < 4112u) { seg = 1; off = idx - 16u; }
  else if (idx < 1052688u) { seg = 2; off = idx - 4112u; }
  else { seg = 3; off = idx - 1052688u; }
  const uint32_t flags = ((raw >> 29) & 1u) << 4 | ((raw >> 30) & 1u) << 5 | seg << 6;
  out[0] = (uint8_t)((off >> (8 * seg)) | flags);
  for (uint32_t b = 1; b <= seg; ++b) out[b] = (uint8_t)(off >> (8 * (seg - b)));
  return seg + 1;
}

__global__ void __launch_bounds__(SER_THREADS)
node_tile_bytes_kernel(const uint2* __restrict__ nodes, uint32_t n, unsigned long long* __restrict__ tile_bytes) {
  __shared__ uint32_t sm[SER_THREADS / 32];
  uint32_t mine = 0;
  const uint32_t first = blockIdx.x * SER_TILE + threadIdx.x * SER_PER_THREAD;
#pragma unroll
  for (int j = 0; j < SER_PER_THREAD; ++j)
    if (first + j < n) {
      const uint2 nd = __ldg(nodes + first + j);
      mine += ptr_len(nd.x) + ptr_len(nd.y);
    }
  uint32_t total;
  block_exclusive_sum<SER_THREADS>(mine, sm, &total);
  if (threadIdx.x == 0) tile_bytes[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SER_THREADS)
emit_nodes_kernel(const uint2* __restrict__ nodes, uint32_t n, const unsigned long long* __restrict__ tile_off,
                  uint8_t* __restrict__ out, unsigned long long layer_base) {
  __shared__ uint32_t sm[SER_THREADS / 32];
  __shared__ __align__(16) uint8_t stage[SER_TILE * 8 + 16];
  const unsigned long long dst = layer_base + tile_off[blockIdx.x];
  const uint32_t shift = (uint32_t)(dst & 3ull);
  uint2 nd[SER_PER_THREAD];
  uint32_t mine = 0;
  const uint32_t first = blockIdx.x * SER_TILE + threadIdx.x * SER_PER_THREAD;
#pragma unroll
  for (int j = 0; j < SER_PER_THREAD; ++j) {
    nd[j] = make_uint2(0, 0);
    if (first + j < n) {
      nd[j] = __ldg(nodes + first + j);
      mine += ptr_len(nd[j].x) + ptr_len(nd[j].y);
    }
  }
  uint32_t total;
  uint32_t o = shift + block_exclusive_sum<SER_THREADS>(mine, sm, &total);
#pragma unroll
  for (int j = 0; j < SER_PER_THREAD; ++j)
    if (first + j < n) {
      o += ptr_encode(nd[j].x, stage + o);
      o += ptr_encode(nd[j].y, stage + o);
    }
  __syncthreads();
  copy_out_staged<SER_THREADS>(reinterpret_cast<char*>(out) + (dst - shift), stage, shift, total);
}

// leaves: low ceil(S/2) bytes of the word, most significant first (src/dna.cpp:149-151)
__global__ void __launch_bounds__(SER_THREADS)
emit_leaves_kernel(const unsigned long long* __restrict__ leaves, uint32_t n, int leaf_bytes, uint8_t* __restrict__ out,
                   unsigned long long base) {
  __shared__ __align__(16) uint8_t stage[SER_TILE * 8 + 16];
  const uint32_t tile_first = blockIdx.x * SER_TILE;
  const uint32_t here = min((uint32_t)SER_TILE, n - tile_first);
  const unsigned long long dst = base + (unsigned long long)tile_first * leaf_bytes;
  const uint32_t shift = (uint32_t)(dst & 3ull);
#pragma unroll
  for (int it = 0; it < SER_PER_THREAD; ++it) {
    const uint32_t j = it * SER_THREADS + threadIdx.x;
    if (j < here) {
      const unsigned long long v = __ldg(leaves + tile_first + j);
      uint8_t* o = stage + shift + j * leaf_bytes;
      for (int b = 0; b < leaf_bytes; ++b) o[b] = (uint8_t)(v >> (8 * (leaf_bytes - 1 - b)));
    }
  }
  __syncthreads();
  copy_out_staged<SER_THREADS>(reinterpret_cast<char*>(out) + (dst - shift), stage, shift, here * leaf_bytes);
}

struct Header {
  unsigned long long off, value;
  uint32_t bytes, pad;
};
__global__ void emit_headers_kernel(const Header* __restrict__ h, uint32_t n, uint8_t* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Header hd = h[i];
  for (uint32_t b = 0; b < hd.bytes; ++b) out[hd.off + b] = (uint8_t)(hd.value >> (8 * (hd.bytes - 1 - b)));
}

// ---- host --------------------------------------------------------------------------

int stream_plan(Tree& t) {
  if (!t.built) return t.fail(STB_ERR_NOT_BUILT, "tree is empty");
  if (t.plan_valid) return STB_OK;
  cudaStream_t st = t.stream;
  const size_t L = t.layers.size();
  t.layer_tile_off.clear();
  t.layer_tile_off.resize(L);
  DevBuf<unsigned long long> totals;
  STB_CUDA(t, totals.alloc(L, st));
  for (size_t k = 0; k < L; ++k) {
    const uint32_t n = (uint32_t)t.layers[k].count;
    const uint32_t tiles = (uint32_t)ceil_div(n, SER_TILE);
    STB_CUDA(t, t.layer_tile_off[k].alloc(tiles, st));
    {
      Launch l(t, "node_tile_bytes");
      node_tile_bytes_kernel<<<tiles, SER_THREADS, 0, st>>>(t.layers[k].nodes.ptr, n, t.layer_tile_off[k].ptr);
    }
    {
      Launch l(t, "scan_tile_bytes");
      exclusive_scan_rows_kernel<<<1, 1024, 0, st>>>(t.layer_tile_off[k].ptr, tiles, totals.ptr + k);
    }
  }
  std::vector<unsigned long long> h(L);
  STB_CUDA(t, cudaMemcpyAsync(h.data(), totals.ptr, L * 8, cudaMemcpyDeviceToHost, st));
  STB_CUDA(t, cudaStreamSynchronize(st));
  STB_CUDA(t, cudaGetLastError());
  t.layer_stream_bytes.assign(h.begin(), h.end());
  uint64_t total = ptr_len(t.root) + 8 + t.n_leaves * (uint64_t)((t.S + 1) / 2);
  for (size_t k = 0; k < L; ++k) total += 8 + t.layer_stream_bytes[k];
  t.stream_bytes = total;
  t.plan_valid = true;
  return STB_OK;
}

int serialize_tree(Tree& t, uint8_t* d_out, uint64_t cap) {
  STB_TRY(stream_plan(t));
  if (cap < t.stream_bytes) return t.fail(STB_ERR_BUFFER_TOO_SMALL, "serialize: buffer smaller than bytes()");
  for (const auto& layer : t.layers)
    if (layer.count > 1052688ull + 0xfffffffull)
      return t.fail(STB_ERR_INDEX_CEILING, "a layer is too large for the 28-bit pointer offset");
  if (t.n_leaves > 1052688ull + 0xfffffffull)
    return t.fail(STB_ERR_INDEX_CEILING, "leaf table is too large for the 28-bit pointer offset");
  cudaStream_t st = t.stream;
  const int leaf_bytes = (t.S + 1) / 2;
  std::vector<Header> headers;
  uint8_t rootb[4];
  const uint32_t rlen = ptr_encode(t.root, rootb);
  unsigned long long rootv = 0;
  for (uint32_t b = 0; b < rlen; ++b) rootv = (rootv << 8) | rootb[b];
  uint64_t off = 0;
  headers.push_back(Header{off, rootv, rlen, 0});
  off += rlen;
  headers.push_back(Header{off, t.n_leaves, 8, 0});
  off += 8;
  const uint64_t leaves_base = off;
  off += t.n_leaves * (uint64_t)leaf_bytes;
  std::vector<uint64_t> layer_base(t.layers.size());
  for (size_t k = 0; k < t.layers.size(); ++k) {
    headers.push_back(Header{off, t.layers[k].count, 8, 0});
    off += 8;
    layer_base[k] = off;
    off += t.layer_stream_bytes[k];
  }
  DevBuf<Header> d_headers;
  STB_CUDA(t, d_headers.alloc(headers.size(), st));
  STB_CUDA(t, cudaMemcpyAsync(d_headers.ptr, headers.data(), headers.size() * sizeof(Header), cudaMemcpyHostToDevice, st));
  {
    Launch l(t, "emit_headers");
    emit_headers_kernel<<<(unsigned)ceil_div(headers.size(), 64), 64, 0, st>>>(d_headers.ptr, (uint32_t)headers.size(), d_out);
  }
  if (t.n_leaves) {
    Launch l(t, "emit_leaves");
    emit_leaves_kernel<<<(unsigned)ceil_div(t.n_leaves, SER_TILE), SER_THREADS, 0, st>>>(t.leaves.ptr, (uint32_t)t.n_leaves, leaf_bytes, d_out, leaves_base);
  }
  for (size_t k = 0; k < t.layers.size(); ++k) {
    const uint32_t n = (uint32_t)t.layers[k].count;
    Launch l(t, "emit_nodes");
    emit_nodes_kernel<<<(unsigned)ceil_div(n, SER_TILE), SER_THREADS, 0, st>>>(t.layers[k].nodes.ptr, n, t.layer_tile_off[k].ptr, d_out, layer_base[k]);
  }
  STB_CUDA(t, cudaStreamSynchronize(st));  // headers vector must outlive the copy
  STB_CUDA(t, cudaGetLastError());
  return STB_OK;
}

// ---- deserialize: the variable-length stream parsed on the device ----------------------------------
// A pointer's length is known only from its first byte, so where the pointers of a layer start looks
// sequential.  It is a 4-state automaton, though: seen from a 32-byte chunk, the only unknown is
// where the first pointer of the chunk starts (offset 0..3: a pointer spans at most 4 bytes), and every
// entry offset maps to an exit offset into the next chunk and a number of pointers.  Such maps compose
// associatively, so: pass 1 reduces every 8 KiB tile to its map, one CTA scans the tile maps (which also
// numbers the pointers), pass 2 walks every chunk from its now known entry, decodes the pointers and
// writes them out by number.  A layer's byte length is not in the stream (only its node count), so a
// layer is parsed over the longest extent it could have (8 bytes per node) and the thread that decodes
// its last pointer reports where the layer really ends; the host reads that number and goes on.
constexpr int DP_THREADS = 256;
constexpr int DP_CHUNK = 32;                      // bytes per thread
constexpr int DP_TILE = DP_THREADS * DP_CHUNK;    // bytes per CTA
constexpr uint64_t DP_SMALL = 2048;               // layers of at most this many nodes are parsed on the host

struct ParseMap {
  uint32_t exits;   // 2 bits per entry offset: the offset at which the next chunk's first pointer starts
  uint32_t cnt[4];  // pointers that start inside, per entry offset
};

__device__ __forceinline__ uint32_t pick4(const uint32_t (&v)[4], uint32_t i) {
  return i == 0 ? v[0] : (i == 1 ? v[1] : (i == 2 ? v[2] : v[3]));
}

// `a` first, then `b`
__device__ __forceinline__ ParseMap compose(const ParseMap& a, const ParseMap& b) {
  ParseMap r;
  r.exits = 0;
#pragma unroll
  for (uint32_t e = 0; e < 4; ++e) {
    const uint32_t x = (a.exits >> (2 * e)) & 3u;
    r.exits |= ((b.exits >> (2 * x)) & 3u) << (2 * e);
    r.cnt[e] = a.cnt[e] + pick4(b.cnt, x);
  }
  return r;
}

__device__ __forceinline__ ParseMap shfl_up_map(const ParseMap& m, int d) {
  ParseMap r;
  r.exits = __shfl_up_sync(0xffffffffu, m.exits, d);
#pragma unroll
  for (int e = 0; e < 4; ++e) r.cnt[e] = __shfl_up_sync(0xffffffffu, m.cnt[e], d);
  return r;
}

__device__ __forceinline__ ParseMap identity_map() { return ParseMap{0xE4u, {0u, 0u, 0u, 0u}}; }  // exits[e] = e

// The tile's bytes in shared memory, transposed: word w of thread t's chunk at sw[w * DP_THREADS + t]
// (a thread walking its chunk then never shares a bank with another), plus the first word after the tile.
struct TileBytes {
  uint32_t* sw;
  __device__ __forceinline__ uint32_t word(uint32_t t, uint32_t w) const {
    return w < 8u ? sw[w * DP_THREADS + t] : sw[t + 1u < (uint32_t)DP_THREADS ? t + 1u : 8u * DP_THREADS];
  }
  __device__ __forceinline__ uint32_t byte(uint32_t t, uint32_t pos) const { return (word(t, pos >> 2) >> (8u * (pos & 3u))) & 0xffu; }
};

__device__ __forceinline__ void load_tile(const uint8_t* __restrict__ stream, uint64_t tile_begin, uint32_t* sw) {
  const uint32_t t = threadIdx.x;
  const uint4* src = reinterpret_cast<const uint4*>(stream + tile_begin + (uint64_t)t * DP_CHUNK);
  const uint4 a = __ldg(src), b = __ldg(src + 1);
  sw[0 * DP_THREADS + t] = a.x; sw[1 * DP_THREADS + t] = a.y; sw[2 * DP_THREADS + t] = a.z; sw[3 * DP_THREADS + t] = a.w;
  sw[4 * DP_THREADS + t] = b.x; sw[5 * DP_THREADS + t] = b.y; sw[6 * DP_THREADS + t] = b.z; sw[7 * DP_THREADS + t] = b.w;
  if (t == 0) sw[8 * DP_THREADS] = __ldg(reinterpret_cast<const uint32_t*>(stream + tile_begin + DP_TILE));
}

// the chunk of thread t as a map; the layer's first chunk starts at `start_off` whatever the entry
__device__ __forceinline__ ParseMap chunk_map(const TileBytes& tb, uint32_t t, bool first_chunk, uint32_t start_off) {
  ParseMap m;
  m.exits = 0;
#pragma unroll
  for (uint32_t e = 0; e < 4; ++e) {
    uint32_t pos = first_chunk ? start_off : e, c = 0;
    while (pos < (uint32_t)DP_CHUNK) {
      pos += 1u + (tb.byte(t, pos) >> 6);
      ++c;
    }
    m.exits |= (pos - DP_CHUNK) << (2 * e);
    m.cnt[e] = c;
  }
  return m;
}

// inclusive scan over the CTA's 256 chunk maps; returns the exclusive map of this thread, the tile's in *tile
__device__ __forceinline__ ParseMap block_scan_maps(const ParseMap& mine, ParseMap* warp_maps /* shared, 8 */, ParseMap* tile) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ParseMap incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const ParseMap up = shfl_up_map(incl, d);
    if (lane >= (uint32_t)d) incl = compose(up, incl);
  }
  if (lane == 31) warp_maps[warp] = incl;
  __syncthreads();
  ParseMap before = identity_map(), total = identity_map();
  for (uint32_t w = 0; w < DP_THREADS / 32; ++w) {
    if (w == warp) before = total;
    total = compose(total, warp_maps[w]);
  }
  *tile = total;
  ParseMap excl = shfl_up_map(incl, 1);
  if (lane == 0) excl = identity_map();
  __syncthreads();
  return compose(before, excl);
}

__global__ void __launch_bounds__(DP_THREADS)
parse_tile_maps_kernel(const uint8_t* __restrict__ stream, uint64_t begin, uint32_t start_off, ParseMap* __restrict__ tile_maps) {
  __shared__ uint32_t sw[8 * DP_THREADS + 1];
  __shared__ ParseMap warp_maps[DP_THREADS / 32];
  load_tile(stream, begin + (uint64_t)blockIdx.x * DP_TILE, sw);
  __syncthreads();
  const TileBytes tb{sw};
  const ParseMap mine = chunk_map(tb, threadIdx.x, blockIdx.x == 0 && threadIdx.x == 0, start_off);
  ParseMap tile;
  block_scan_maps(mine, warp_maps, &tile);
  if (threadIdx.x == 0) tile_maps[blockIdx.x] = tile;
}

// exclusive scan of the tile maps, evaluated at entry offset 0: per tile (entry offset, pointers before it)
__global__ void __launch_bounds__(1024)
parse_scan_tiles_kernel(const ParseMap* __restrict__ tile_maps, uint32_t tiles, uint2* __restrict__ tile_entry) {
  __shared__ ParseMap warp_maps[32];
  __shared__ uint32_t carry_state;
  __shared__ unsigned long long carry_cnt;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    carry_state = 0u;
    carry_cnt = 0ull;
  }
  __syncthreads();
  for (uint32_t base = 0; base < tiles; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    const ParseMap mine = i < tiles ? tile_maps[i] : identity_map();
    ParseMap incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const ParseMap up = shfl_up_map(incl, d);
      if (lane >= (uint32_t)d) incl = compose(up, incl);
    }
    if (lane == 31) warp_maps[warp] = incl;
    __syncthreads();
    if (warp == 0) {  // inclusive scan of the 32 warp totals
      ParseMap w = warp_maps[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const ParseMap up = shfl_up_map(w, d);
        if (lane >= (uint32_t)d) w = compose(up, w);
      }
      warp_maps[lane] = w;
    }
    __syncthreads();
    const ParseMap before = warp ? warp_maps[warp - 1] : identity_map(), total = warp_maps[31];
    ParseMap excl = shfl_up_map(incl, 1);
    if (lane == 0) excl = identity_map();
    excl = compose(before, excl);
    const uint32_t st = carry_state;
    const unsigned long long cn = carry_cnt;
    if (i < tiles) {
      const unsigned long long prefix = cn + pick4(excl.cnt, st);
      tile_entry[i] = make_uint2((excl.exits >> (2 * st)) & 3u, (uint32_t)(prefix < 0xffffffffull ? prefix : 0xffffffffull));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      carry_state = (total.exits >> (2 * st)) & 3u;
      carry_cnt = cn + pick4(total.cnt, st);
    }
    __syncthreads();
  }
}

__device__ __forceinline__ uint32_t ptr_decode(uint32_t b0, uint32_t rest /* the following bytes, first in the low byte */) {
  const uint32_t seg = b0 >> 6;
  uint32_t off = b0 & 0xfu;
  for (uint32_t b = 0; b < seg; ++b) off = (off << 8) | ((rest >> (8 * b)) & 0xffu);
  const uint32_t first[4] = {0u, 16u, 4112u, 1052688u};
  const uint32_t idx = (seg == 3u && off == 0xfffffffu) ? IDX_MASK : pick4(first, seg) + off;
  return idx | (((b0 >> 4) & 1u) << 29) | (((b0 >> 5) & 1u) << 30);
}

// A decoded child pointer the tree cannot follow: an index past the layer below, or the null index with the
// mirror or transpose bit set (ptr_is_null does not count that as null, so it would be followed to index 2^29-1).
__host__ __device__ __forceinline__ bool ptr_unfollowable(uint32_t raw, uint32_t below) {
  const uint32_t idx = raw & IDX_MASK;
  return idx == IDX_MASK ? (raw & (MIRROR | TRANSPOSE)) != 0u : idx >= below;
}

// result[0] = absolute offset of the byte after the layer's last pointer, result[1] = 1 when a pointer cannot be
// followed (ptr_unfollowable)
__global__ void __launch_bounds__(DP_THREADS)
parse_emit_kernel(const uint8_t* __restrict__ stream, uint64_t begin, uint32_t start_off, const uint2* __restrict__ tile_entry,
                  uint32_t* __restrict__ out, uint32_t n_ptrs, uint32_t below, unsigned long long* __restrict__ result) {
  __shared__ uint32_t sw[8 * DP_THREADS + 1];
  __shared__ ParseMap warp_maps[DP_THREADS / 32];
  __shared__ uint32_t sout[DP_TILE];
  const uint2 entry = tile_entry[blockIdx.x];
  if (entry.y >= n_ptrs) return;  // past the layer's end
  const uint64_t tile_begin = begin + (uint64_t)blockIdx.x * DP_TILE;
  load_tile(stream, tile_begin, sw);
  __syncthreads();
  const TileBytes tb{sw};
  const uint32_t t = threadIdx.x;
  const bool first_chunk = blockIdx.x == 0 && t == 0;
  const ParseMap mine = chunk_map(tb, t, first_chunk, start_off);
  ParseMap tile;
  const ParseMap excl = block_scan_maps(mine, warp_maps, &tile);
  const uint32_t e = (excl.exits >> (2 * entry.x)) & 3u;
  uint32_t local = pick4(excl.cnt, entry.x);           // pointers of the tile before this chunk
  const uint32_t tile_total = pick4(tile.cnt, entry.x);
  uint32_t pos = first_chunk ? start_off : e;
  bool bad = false;
  while (pos < (uint32_t)DP_CHUNK) {
    const uint32_t b0 = tb.byte(t, pos);
    const uint32_t seg = b0 >> 6;
    uint32_t rest = 0;
    for (uint32_t b = 0; b < seg; ++b) rest |= tb.byte(t, pos + 1 + b) << (8 * b);
    const uint32_t raw = ptr_decode(b0, rest);
    const uint32_t number = entry.y + local;  // < 2^32: entry.y < n_ptrs <= 2^30, local <= 8192
    pos += seg + 1u;
    if (number < n_ptrs) {
      bad |= ptr_unfollowable(raw, below);
      sout[local] = raw;
      if (number == n_ptrs - 1u) result[0] = tile_begin + (uint64_t)t * DP_CHUNK + pos;
    }
    ++local;
  }
  if (bad) result[1] = 1ull;
  __syncthreads();
  const uint32_t keep = min(tile_total, n_ptrs - entry.y);
  for (uint32_t i = t; i < keep; i += DP_THREADS) out[entry.y + i] = sout[i];
}

// leaves: ceil(S/2) bytes each, most significant first (src/dna.cpp:149-161)
__global__ void __launch_bounds__(256)
parse_leaves_kernel(const uint8_t* __restrict__ stream, uint64_t begin, uint32_t n, int leaf_bytes, unsigned long long* __restrict__ leaves) {
  const uint32_t i = blockIdx.x * 256 + threadIdx.x;
  if (i >= n) return;
  const uint8_t* p = stream + begin + (uint64_t)i * leaf_bytes;
  unsigned long long v = 0;
  for (int b = 0; b < leaf_bytes; ++b) v = (v << 8) | __ldg(p + b);
  leaves[i] = v;
}

// shared_tree::deserialize, src/shared_tree.cpp:520-538; pointers come back with invariant = false (:162).
// The stream is copied to the device once; the layers are parsed there (see above), the small top of the
// tree on the host.  A foreign or damaged stream must not make the device follow wild indices (an illegal
// address is sticky for the whole process).  The reference trusts its input; here STB_ERR_BAD_STREAM rejects:
//   - a stream that ends inside the header, the leaf table or a node;
//   - no leaves, a node layer of no nodes, or no node layer at all;
//   - a leaf table or a layer too large for the pointer format to index;
//   - a child pointer that indexes past the layer below, or the null index with the mirror or transpose bit set;
//   - a root that does not index the top layer (a null root included);
//   - a right edge that leads into a null: the node the width walk reaches has no child to go on with
//     (compute_width).  Nulls elsewhere are read as they are; builds write them nowhere else.
int deserialize_tree(Tree& t, const uint8_t* in, uint64_t len) {
  static const uint32_t start[4] = {0u, 16u, 4112u, 1052688u};
  t.clear();
  cudaStream_t st = t.stream;
  uint64_t o = 0;
  auto read_ptr = [&](uint32_t& raw) -> bool {
    if (o >= len) return false;
    const uint32_t b0 = in[o];
    const uint32_t seg = (b0 >> 6) & 3u;
    if (o + seg + 1 > len) return false;
    uint32_t off = b0 & 0xfu;
    for (uint32_t b = 1; b <= seg; ++b) off = (off << 8) | in[o + b];
    o += seg + 1;
    const uint32_t idx = (seg == 3 && off == 0xfffffffu) ? IDX_MASK : start[seg] + off;
    raw = idx | (((b0 >> 4) & 1u) << 29) | (((b0 >> 5) & 1u) << 30);
    return true;
  };
  auto read_u64 = [&](uint64_t& v) -> bool {
    if (o + 8 > len) return false;
    v = 0;
    for (int b = 0; b < 8; ++b) v = (v << 8) | in[o + b];
    o += 8;
    return true;
  };
  uint32_t root;
  uint64_t n_leaves;
  if (!read_ptr(root) || !read_u64(n_leaves)) return t.fail(STB_ERR_BAD_STREAM, "stream ends inside the header");
  const int leaf_bytes = (t.S + 1) / 2;
  if (n_leaves > (len - o) / (uint64_t)leaf_bytes) return t.fail(STB_ERR_BAD_STREAM, "stream ends inside the leaf table");
  if (n_leaves >= IDX_MASK) return t.fail(STB_ERR_BAD_STREAM, "leaf table larger than the pointer format can index");
  if (n_leaves == 0) return t.fail(STB_ERR_BAD_STREAM, "stream holds no leaves");

  // the whole stream on the device (the handle's grow-only staging buffer), zero-padded by one tile
  const uint64_t padded = ((len + 31) & ~31ull) + DP_TILE + 64;
  STB_CUDA(t, t.staging.ensure(padded, st));
  uint8_t* d_stream = reinterpret_cast<uint8_t*>(t.staging.ptr);
  // copied in chunks on a second stream; a layer is parsed as soon as the chunks it can reach have arrived, so the
  // parse (about a third of the copy's time) hides behind the copy
  constexpr uint64_t COPY_CHUNK = 64ull << 20;
  const uint64_t chunks = ceil_div(len, COPY_CHUNK);
  STB_CUDA(t, t.copy_lane(chunks + 1));
  STB_CUDA(t, cudaEventRecord(t.copy_events[chunks], st));  // the staging buffer is free (and allocated) at this point of `st`
  STB_CUDA(t, cudaStreamWaitEvent(t.copy_stream, t.copy_events[chunks], 0));
  for (uint64_t c = 0; c < chunks; ++c) {
    const uint64_t at = c * COPY_CHUNK, n = std::min<uint64_t>(COPY_CHUNK, len - at);
    STB_CUDA(t, cudaMemcpyAsync(d_stream + at, in + at, n, cudaMemcpyHostToDevice, t.copy_stream));
    STB_CUDA(t, cudaEventRecord(t.copy_events[c], t.copy_stream));
  }
  STB_CUDA(t, cudaMemsetAsync(d_stream + len, 0, padded - len, st));
  // a damaged stream is reported only after the copies have ended: the caller's buffer must be free when a call returns
  auto bad = [&](const std::string& what) {
    cudaStreamSynchronize(t.copy_stream);
    return t.fail(STB_ERR_BAD_STREAM, what);
  };
  int64_t waited = -1;
  auto wait_for = [&](uint64_t end_byte) -> cudaError_t {  // `st` goes on once bytes [0, end_byte) are on the device
    const int64_t c = (int64_t)std::min<uint64_t>(chunks - 1, (std::max<uint64_t>(end_byte, 1) - 1) / COPY_CHUNK);
    if (c <= waited) return cudaSuccess;
    waited = c;
    return cudaStreamWaitEvent(st, t.copy_events[c], 0);
  };

  STB_CUDA(t, t.leaves.alloc(n_leaves, st));
  STB_CUDA(t, wait_for(o + n_leaves * (uint64_t)leaf_bytes));
  if (n_leaves) {
    Launch l(t, "parse_leaves");
    parse_leaves_kernel<<<(unsigned)ceil_div(n_leaves, 256), 256, 0, st>>>(d_stream, o, (uint32_t)n_leaves, leaf_bytes, t.leaves.ptr);
  }
  o += n_leaves * (uint64_t)leaf_bytes;

  DevBuf<ParseMap> tile_maps;
  DevBuf<uint2> tile_entry;
  DevBuf<unsigned long long> result;
  STB_CUDA(t, result.alloc(2, st));
  uint64_t below = n_leaves;
  while (o + 8 <= len) {  // layers until the stream ends (:528-530)
    uint64_t count;
    read_u64(count);
    if (count > (len - o) / 2) return bad("layer size exceeds the remaining stream");
    if (count >= IDX_MASK) return bad("layer larger than the pointer format can index");
    const size_t k = t.layers.size();
    if (count == 0) return bad("node layer " + std::to_string(k) + " holds no nodes");
    t.layers.emplace_back();
    Layer& layer = t.layers.back();
    layer.count = count;
    STB_CUDA(t, layer.nodes.alloc(count, st));
    if (count <= DP_SMALL) {  // the top of the tree: a few kilobytes, not worth three launches and a read-back
      std::vector<uint2> nodes(count);
      for (uint64_t i = 0; i < count; ++i) {
        uint2 nd;
        if (!read_ptr(nd.x) || !read_ptr(nd.y)) return bad("stream ends inside a node");
        if (ptr_unfollowable(nd.x, (uint32_t)below) || ptr_unfollowable(nd.y, (uint32_t)below))
          return bad("a node of layer " + std::to_string(k) + " points past the end of the layer below or holds a flagged null");
        nodes[i] = nd;
      }
      STB_CUDA(t, cudaMemcpyAsync(layer.nodes.ptr, nodes.data(), count * sizeof(uint2), cudaMemcpyHostToDevice, st));
      STB_CUDA(t, cudaStreamSynchronize(st));  // `nodes` is about to go away
    } else {
      const uint64_t begin = o & ~31ull;
      const uint32_t start_off = (uint32_t)(o - begin);
      const uint64_t extent = std::min<uint64_t>(len - begin, start_off + 8 * count);  // the longest the layer can be
      const uint32_t tiles = (uint32_t)ceil_div(extent, DP_TILE);
      STB_CUDA(t, wait_for(std::min<uint64_t>(len, begin + (uint64_t)tiles * DP_TILE + 64)));
      STB_CUDA(t, tile_maps.ensure(tiles, st));
      STB_CUDA(t, tile_entry.ensure(tiles, st));
      STB_CUDA(t, cudaMemsetAsync(result.ptr, 0, 16, st));
      {
        Launch l(t, "parse_tile_maps");
        parse_tile_maps_kernel<<<tiles, DP_THREADS, 0, st>>>(d_stream, begin, start_off, tile_maps.ptr);
      }
      {
        Launch l(t, "parse_scan_tiles");
        parse_scan_tiles_kernel<<<1, 1024, 0, st>>>(tile_maps.ptr, tiles, tile_entry.ptr);
      }
      {
        Launch l(t, "parse_emit");
        parse_emit_kernel<<<tiles, DP_THREADS, 0, st>>>(d_stream, begin, start_off, tile_entry.ptr, reinterpret_cast<uint32_t*>(layer.nodes.ptr),
                                                        (uint32_t)(2 * count), (uint32_t)below, result.ptr);
      }
      unsigned long long res[2] = {0, 0};
      STB_CUDA(t, cudaMemcpyAsync(res, result.ptr, 16, cudaMemcpyDeviceToHost, st));
      STB_CUDA(t, cudaStreamSynchronize(st));
      STB_CUDA(t, cudaGetLastError());
      if (res[0] == 0 || res[0] > len) return bad("stream ends inside a node");
      if (res[1]) return bad("a node of layer " + std::to_string(k) + " points past the end of the layer below or holds a flagged null");
      o = res[0];
    }
    below = count;
  }
  STB_CUDA(t, wait_for(len));  // the caller's buffer is free again when this call returns
  STB_CUDA(t, cudaStreamSynchronize(st));
  if (t.layers.empty()) return bad("stream holds no node layer");
  if ((root & IDX_MASK) >= below) return bad("the root pointer does not index the top layer");
  t.n_leaves = n_leaves;
  t.root = root;
  t.built = true;
  t.plan_valid = false;
  return compute_width(t);
}

}  // namespace stb
