// capi.cu — the extern "C" boundary declared in include/shared_tree_b200.h.
#include <algorithm>
#include <cstring>
#include <new>

#include "tree.h"

namespace stb {

uint64_t g_kernel_launches = 0;

cudaEvent_t Ctx::get_event() {
  if (!event_pool.empty()) {
    cudaEvent_t e = event_pool.back();
    event_pool.pop_back();
    return e;
  }
  cudaEvent_t e;
  cudaEventCreate(&e);
  return e;
}

void Ctx::flush_profile() {
  if (pending.empty()) return;
  cudaStreamSynchronize(stream);
  for (auto& p : pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
      Acc& a = account(p.name, p.level);
      a.ms += ms;
      a.launches += 1;
    }
    event_pool.push_back(p.a);
    event_pool.push_back(p.b);
  }
  pending.clear();
}

Ctx::Acc& Ctx::account(const char* name, int level) {
  const std::string key = level >= 0 ? std::string(name) + "@L" + std::to_string(level) : std::string(name);
  auto it = acc.find(key);
  if (it == acc.end()) {
    acc_order.push_back(key);
    it = acc.emplace(key, Acc{}).first;
  }
  return it->second;
}

cudaError_t Ctx::copy_lane(size_t events) {
  if (!copy_stream) {
    const cudaError_t e = cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) return e;
  }
  while (copy_events.size() < events) {
    cudaEvent_t ev;
    const cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return e;
    copy_events.push_back(ev);
  }
  return cudaSuccess;
}

Ctx::~Ctx() {
  for (auto e : copy_events) cudaEventDestroy(e);
  if (copy_stream) cudaStreamDestroy(copy_stream);
  for (auto& p : pending) {
    cudaEventDestroy(p.a);
    cudaEventDestroy(p.b);
  }
  for (auto e : event_pool) cudaEventDestroy(e);
}

__global__ void needs_extraction_kernel(const char* __restrict__ text, unsigned long long len, uint32_t* flag) {
  // any newline, or a header at the very start, means the text is not a bare body
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x * 16ull;
  bool found = false;
  for (unsigned long long i = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 16ull; i < len && !found; i += stride) {
    if (i + 16 <= len) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(text + i));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t x = w[k] ^ 0x0a0a0a0au;  // zero byte <=> '\n'
        if ((x - 0x01010101u) & ~x & 0x80808080u) found = true;
      }
    } else {
      for (unsigned long long j = i; j < len; ++j)
        if (text[j] == '\n') found = true;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && len && text[0] == '>') found = true;
  if (found) *flag = 1u;
}

}  // namespace stb

using namespace stb;

namespace {

int use_device(const Tree* t) {
  const cudaError_t e = cudaSetDevice(t->device);
  if (e != cudaSuccess) return t->fail_cuda(e, "cudaSetDevice", __FILE__, __LINE__);
  return STB_OK;
}

// Brings `count` elements of T onto the device (16-byte aligned) when they are not
// already there.  `hold` owns the temporary copy.
template <typename T>
int to_device(Tree& t, const T* src, uint64_t count, int memory, DevBuf<T>& hold, const T** out) {
  if (memory == STB_DEVICE && (reinterpret_cast<uintptr_t>(src) & 15u) == 0) {
    *out = src;
    return STB_OK;
  }
  // the handle's grow-only staging buffer: no device allocation per call in steady state
  (void)hold;
  STB_CUDA(t, t.staging.ensure(count * sizeof(T) + 16, t.stream));
  T* dst = reinterpret_cast<T*>(t.staging.ptr);
  if (count) {
    Launch l(t, memory == STB_HOST ? "h2d_copy" : "d2d_copy", false);
    STB_CUDA(t, cudaMemcpyAsync(dst, src, count * sizeof(T),
                                memory == STB_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, t.stream));
  }
  *out = dst;
  return STB_OK;
}

template <typename T>
int from_device(Tree& t, T* dst, const T* d_src, uint64_t count, int memory) {
  if (count == 0) return STB_OK;
  Launch l(t, memory == STB_HOST ? "d2h_copy" : "d2d_copy", false);
  STB_CUDA(t, cudaMemcpyAsync(dst, d_src, count * sizeof(T),
                              memory == STB_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, t.stream));
  STB_CUDA(t, cudaStreamSynchronize(t.stream));
  return STB_OK;
}

bool valid_memory(int m) { return m == STB_HOST || m == STB_DEVICE; }

}  // namespace

extern "C" {

int stb_create(stb_tree** out, int device, int dna_size, void* cuda_stream) {
  if (!out) return STB_ERR_INVALID_ARG;
  *out = nullptr;
  if (dna_size < 1 || dna_size > 16) return STB_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return STB_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return STB_ERR_CUDA;
  // keep freed blocks in the stream-ordered pool: levels re-allocate the same sizes
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t threshold = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
  }
  stb_tree* t = new (std::nothrow) stb_tree();
  if (!t) return STB_ERR_INVALID_ARG;
  t->device = device;
  t->S = dna_size;
  t->stream = (cudaStream_t)cuda_stream;
  *out = t;
  return STB_OK;
}

static uint64_t* option_slot(Options& o, const char* name) {
  const struct { const char* name; uint64_t* slot; } table[] = {
      {"bucket_min", &o.bucket_min}, {"bucket_levels", &o.bucket_levels}, {"bucket_cap", &o.bucket_cap}, {"partition_threads", &o.partition_threads}, {"dedup_threads", &o.dedup_threads}, {"bucket_slack_permille", &o.bucket_slack_permille}, {"bucket_headroom", &o.bucket_headroom},
      {"child_filter", &o.child_filter}, {"locality", &o.locality}, {"coop_max", &o.coop_max}, {"reserve_pipeline", &o.reserve_pipeline}, {"side_table_slots", &o.side_table_slots}, {"profile_levels", &o.profile_levels},
      {"stream_chunk_log2", &o.stream_chunk_log2}, {"stream_min_chunks", &o.stream_min_chunks}, {"leaf_prefix_log2", &o.leaf_prefix_log2},
      {"fused_resolve", &o.fused_resolve}};
  for (const auto& e : table)
    if (std::strcmp(e.name, name) == 0) return e.slot;
  return nullptr;
}

int stb_set_option(stb_tree* tree, const char* name, uint64_t value) {
  if (!tree || !name) return STB_ERR_INVALID_ARG;
  uint64_t* slot = option_slot(tree->opt, name);
  if (!slot) return tree->fail(STB_ERR_INVALID_ARG, std::string("unknown option: ") + name);
  *slot = value;
  return STB_OK;
}

int stb_get_option(const stb_tree* tree, const char* name, uint64_t* value) {
  if (!tree || !name || !value) return STB_ERR_INVALID_ARG;
  const uint64_t* slot = option_slot(const_cast<stb_tree*>(tree)->opt, name);
  if (!slot) return tree->fail(STB_ERR_INVALID_ARG, std::string("unknown option: ") + name);
  *value = *slot;
  return STB_OK;
}

void stb_node_canonical(uint32_t left, uint32_t right, uint32_t* out_left, uint32_t* out_right, uint32_t* out_flags) {
  uint32_t cl, cr, f;
  canonical_node(left, right, cl, cr, f);
  if (out_left) *out_left = cl;
  if (out_right) *out_right = cr;
  if (out_flags) *out_flags = f;
}

uint64_t stb_leaf_canonical(uint64_t leaf, int dna_size, uint32_t* out_flags) {
  uint32_t f;
  const unsigned long long c = canonical_leaf(leaf, dna_size, f);
  if (out_flags) *out_flags = f;
  return c;
}

uint32_t stb_pointer_compose(uint32_t pointer, int mirror, int transpose) { return compose(pointer, mirror ? 1u : 0u, transpose ? 1u : 0u); }

int stb_release_workspace(stb_tree* tree) {
  if (!tree) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  tree->workspace.reset();
  tree->staging.release();
  tree->release_scratch();
  return STB_OK;
}

int stb_destroy(stb_tree* tree) {
  if (!tree) return STB_OK;
  cudaSetDevice(tree->device);
  tree->clear();
  tree->workspace.reset();
  tree->staging.release();
  tree->release_scratch();
  cudaStreamSynchronize(tree->stream);
  delete tree;
  return STB_OK;
}

int stb_clone(const stb_tree* tree, stb_tree** out) {
  if (!tree || !out) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  stb_tree* c = nullptr;
  STB_TRY(stb_create(&c, tree->device, tree->S, tree->stream));
  c->built = tree->built;
  c->n_leaves = tree->n_leaves;
  c->root = tree->root;
  c->width = tree->width;
  c->profiling = tree->profiling;
  c->opt = tree->opt;
  if (tree->built) {
    cudaStream_t st = tree->stream;
    auto fail = [&](cudaError_t e) {
      tree->fail_cuda(e, "clone", __FILE__, __LINE__);
      stb_destroy(c);
      return STB_ERR_CUDA;
    };
    cudaError_t e = c->leaves.alloc(tree->n_leaves, st);
    if (e != cudaSuccess) return fail(e);
    e = cudaMemcpyAsync(c->leaves.ptr, tree->leaves.ptr, tree->n_leaves * 8, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return fail(e);
    for (const auto& layer : tree->layers) {
      c->layers.emplace_back();
      Layer& nl = c->layers.back();
      nl.count = layer.count;
      e = nl.nodes.alloc(layer.count, st);
      if (e != cudaSuccess) return fail(e);
      e = cudaMemcpyAsync(nl.nodes.ptr, layer.nodes.ptr, layer.count * sizeof(uint2), cudaMemcpyDeviceToDevice, st);
      if (e != cudaSuccess) return fail(e);
    }
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(e);
  }
  *out = c;
  return STB_OK;
}

int stb_build_from_body(stb_tree* tree, const char* body, uint64_t len, int memory) {
  if (!tree || (!body && len) || !valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  if (memory == STB_HOST) {  // large host inputs: build chunk by chunk behind the copy
    const int s = build_from_host_body(*tree, body, len);
    if (s != NOT_APPLICABLE) return s;
  }
  DevBuf<char> hold;
  const char* d = nullptr;
  STB_TRY(to_device(*tree, body, len, memory, hold, &d));
  return build_from_body(*tree, d, len);
}

int stb_build_from_fasta(stb_tree* tree, const char* text, uint64_t len, int memory) {
  if (!tree || (!text && len) || !valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  Tree& t = *tree;
  if (len == 0) return t.fail(STB_ERR_EMPTY, "input holds fewer than dna_size bases");
  if (memory == STB_HOST) {  // large host inputs: extract and build chunk by chunk behind the copy
    const int s = build_from_host_fasta(t, text, len);
    if (s != NOT_APPLICABLE) return s;
  }
  DevBuf<char> hold;
  const char* d = nullptr;
  STB_TRY(to_device(t, text, len, memory, hold, &d));
  DevBuf<uint32_t> flag;
  STB_CUDA(t, flag.alloc(1, t.stream));
  STB_CUDA(t, cudaMemsetAsync(flag.ptr, 0, 4, t.stream));
  {
    Launch l(t, "needs_extraction");
    needs_extraction_kernel<<<1184, 256, 0, t.stream>>>(d, len, flag.ptr);
  }
  uint32_t need = 0;
  STB_CUDA(t, cudaMemcpyAsync(&need, flag.ptr, 4, cudaMemcpyDeviceToHost, t.stream));
  STB_CUDA(t, cudaStreamSynchronize(t.stream));
  if (!need) return build_from_body(t, d, len);
  DevBuf<char> body;
  uint64_t body_len = 0;
  STB_TRY(fasta_extract_body(t, d, len, body, &body_len));
  hold.release();
  return build_from_body(t, body.ptr, body_len);
}

int stb_build_from_leaves(stb_tree* tree, const uint64_t* leaves, uint64_t count, int memory) {
  if (!tree || (!leaves && count) || !valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  DevBuf<unsigned long long> hold;
  const unsigned long long* d = nullptr;
  STB_TRY(to_device(*tree, reinterpret_cast<const unsigned long long*>(leaves), count, memory, hold, &d));
  return build_from_leaves(*tree, d, count);
}

int stb_pack_fasta(stb_tree* tree, const char* text, uint64_t len, int text_memory, uint64_t* leaves, uint64_t cap,
                   int leaves_memory, uint64_t* count) {
  if (!tree || (!text && len) || !count || !valid_memory(text_memory) || !valid_memory(leaves_memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  Tree& t = *tree;
  DevBuf<char> hold, body;
  const char* d = nullptr;
  STB_TRY(to_device(t, text, len, text_memory, hold, &d));
  uint64_t body_len = 0;
  STB_TRY(fasta_extract_body(t, d, len, body, &body_len));
  const uint64_t n = body_len / (uint64_t)t.S;
  *count = n;
  if (!leaves) return STB_OK;
  DevBuf<unsigned long long> packed;
  STB_CUDA(t, packed.alloc(n, t.stream));
  STB_TRY(pack_body(t, body.ptr, n, packed.ptr));
  return from_device(t, reinterpret_cast<unsigned long long*>(leaves), packed.ptr, std::min(n, cap), leaves_memory);
}

#define STB_QUERY_PROLOGUE                                         \
  if (!tree || !out) return STB_ERR_INVALID_ARG;                   \
  if (!tree->built) return tree->fail(STB_ERR_NOT_BUILT, "tree is empty");

int stb_depth(const stb_tree* tree, uint64_t* out) {
  STB_QUERY_PROLOGUE
  *out = tree->layers.size() + 1;
  return STB_OK;
}
int stb_width(const stb_tree* tree, uint64_t* out) {
  STB_QUERY_PROLOGUE
  *out = tree->width;
  return STB_OK;
}
int stb_leaf_count(const stb_tree* tree, uint64_t* out) {
  STB_QUERY_PROLOGUE
  *out = tree->n_leaves;
  return STB_OK;
}
int stb_node_count(const stb_tree* tree, uint64_t* out) {
  STB_QUERY_PROLOGUE
  uint64_t s = 0;
  for (const auto& l : tree->layers) s += l.count;
  *out = s;
  return STB_OK;
}
int stb_layer_count(const stb_tree* tree, uint64_t layer, uint64_t* out) {
  STB_QUERY_PROLOGUE
  if (layer >= tree->layers.size()) return tree->fail(STB_ERR_INVALID_ARG, "layer out of range");
  *out = tree->layers[layer].count;
  return STB_OK;
}
int stb_root(const stb_tree* tree, uint32_t* out) {
  STB_QUERY_PROLOGUE
  *out = tree->root;
  return STB_OK;
}
int stb_dna_size(const stb_tree* tree, int* out) {
  if (!tree || !out) return STB_ERR_INVALID_ARG;
  *out = tree->S;
  return STB_OK;
}

int stb_copy_leaves(const stb_tree* tree, uint64_t* out, uint64_t cap, int memory) {
  STB_QUERY_PROLOGUE
  if (!valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  if (cap < tree->n_leaves) return tree->fail(STB_ERR_BUFFER_TOO_SMALL, "copy_leaves: cap < leaf_count()");
  Tree& t = const_cast<stb_tree&>(*tree);
  return from_device(t, reinterpret_cast<unsigned long long*>(out), tree->leaves.ptr, tree->n_leaves, memory);
}

int stb_copy_layer(const stb_tree* tree, uint64_t layer, uint32_t* out, uint64_t cap_nodes, int memory) {
  STB_QUERY_PROLOGUE
  if (!valid_memory(memory)) return STB_ERR_INVALID_ARG;
  if (layer >= tree->layers.size()) return tree->fail(STB_ERR_INVALID_ARG, "layer out of range");
  STB_TRY(use_device(tree));
  const Layer& l = tree->layers[layer];
  if (cap_nodes < l.count) return tree->fail(STB_ERR_BUFFER_TOO_SMALL, "copy_layer: cap < node_count(layer)");
  Tree& t = const_cast<stb_tree&>(*tree);
  return from_device(t, reinterpret_cast<uint2*>(out), l.nodes.ptr, l.count, memory);
}

int stb_histogram(const stb_tree* tree, uint64_t layer, uint64_t* out, uint64_t cap, int memory) {
  STB_QUERY_PROLOGUE
  if (!valid_memory(memory)) return STB_ERR_INVALID_ARG;
  if (layer >= tree->layers.size()) return tree->fail(STB_ERR_INVALID_ARG, "layer out of range");
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  const uint64_t n = layer == 0 ? t.n_leaves : t.layers[layer - 1].count;
  if (cap < n) return t.fail(STB_ERR_BUFFER_TOO_SMALL, "histogram: cap < child layer size");
  if (memory == STB_DEVICE) {
    STB_TRY(histogram_u64(t, layer, reinterpret_cast<unsigned long long*>(out)));
    STB_CUDA(t, cudaStreamSynchronize(t.stream));
    return STB_OK;
  }
  DevBuf<unsigned long long> d;
  STB_CUDA(t, d.alloc(n, t.stream));
  STB_TRY(histogram_u64(t, layer, d.ptr));
  return from_device(t, reinterpret_cast<unsigned long long*>(out), d.ptr, n, STB_HOST);
}

int stb_sort_tree(stb_tree* tree) {
  if (!tree) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  return sort_tree(*tree);
}

int stb_bytes(const stb_tree* tree, uint64_t* out) {
  STB_QUERY_PROLOGUE
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  STB_TRY(stream_plan(t));
  *out = t.stream_bytes;
  return STB_OK;
}

int stb_serialize(const stb_tree* tree, uint8_t* out, uint64_t cap, int memory, uint64_t* written) {
  if (!tree || !out || !valid_memory(memory)) return STB_ERR_INVALID_ARG;
  if (!tree->built) return tree->fail(STB_ERR_NOT_BUILT, "tree is empty");
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  STB_TRY(stream_plan(t));
  if (cap < t.stream_bytes) return t.fail(STB_ERR_BUFFER_TOO_SMALL, "serialize: cap < bytes()");
  if (memory == STB_DEVICE && (reinterpret_cast<uintptr_t>(out) & 3u) == 0) {
    STB_TRY(serialize_tree(t, out, cap));
  } else {
    // through the handle's grow-only staging buffer (the text it held is no longer needed): no 1.7 GB
    // allocation per call
    STB_CUDA(t, t.staging.ensure(t.stream_bytes + 16, t.stream));
    uint8_t* d = reinterpret_cast<uint8_t*>(t.staging.ptr);
    STB_TRY(serialize_tree(t, d, t.stream_bytes));
    STB_TRY(from_device(t, out, d, t.stream_bytes, memory));
  }
  if (written) *written = t.stream_bytes;
  return STB_OK;
}

int stb_deserialize(stb_tree* tree, const uint8_t* bytes, uint64_t len) {
  if (!tree || (!bytes && len)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  return deserialize_tree(*tree, bytes, len);
}

int stb_decode_leaves(const stb_tree* tree, uint64_t first, uint64_t count, uint64_t* out, int memory) {
  STB_QUERY_PROLOGUE
  if (!valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  if (memory == STB_DEVICE) return decode_range(t, first, count, reinterpret_cast<unsigned long long*>(out), nullptr);
  DevBuf<unsigned long long> d;
  STB_CUDA(t, d.alloc(count, t.stream));
  STB_TRY(decode_range(t, first, count, d.ptr, nullptr));
  return from_device(t, reinterpret_cast<unsigned long long*>(out), d.ptr, count, STB_HOST);
}

int stb_decode_ascii(const stb_tree* tree, uint64_t first, uint64_t count, char* out, int memory) {
  STB_QUERY_PROLOGUE
  if (!valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  if (memory == STB_DEVICE) return decode_range(t, first, count, nullptr, out);
  // through the handle's grow-only staging buffer: no allocation of the text's size per call
  STB_CUDA(t, t.staging.ensure(count * (uint64_t)t.S + 16, t.stream));
  STB_TRY(decode_range(t, first, count, nullptr, t.staging.ptr));
  return from_device(t, out, t.staging.ptr, count * (uint64_t)t.S, STB_HOST);
}

int stb_random_access(const stb_tree* tree, const uint64_t* index, uint64_t queries, uint64_t* out, int memory) {
  STB_QUERY_PROLOGUE
  if (!index || !valid_memory(memory)) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  if (memory == STB_DEVICE)
    return random_access(t, reinterpret_cast<const unsigned long long*>(index), queries, reinterpret_cast<unsigned long long*>(out));
  DevBuf<unsigned long long> d_idx, d_out;
  STB_CUDA(t, d_idx.alloc(queries, t.stream));
  STB_CUDA(t, d_out.alloc(queries, t.stream));
  STB_CUDA(t, cudaMemcpyAsync(d_idx.ptr, index, queries * 8, cudaMemcpyHostToDevice, t.stream));
  STB_TRY(random_access(t, d_idx.ptr, queries, d_out.ptr));
  return from_device(t, reinterpret_cast<unsigned long long*>(out), d_out.ptr, queries, STB_HOST);
}

int stb_extract_regions(const stb_tree* tree, const uint64_t* start, const uint64_t* end, const uint8_t* strand,
                        uint64_t n_regions, char* out, uint64_t cap, int memory, uint64_t* written) {
  if (!tree || !written || !valid_memory(memory)) return STB_ERR_INVALID_ARG;
  if (!tree->built) return tree->fail(STB_ERR_NOT_BUILT, "tree is empty");
  if (n_regions == 0) {
    *written = 0;
    return STB_OK;
  }
  if (!start || !end) return tree->fail(STB_ERR_INVALID_ARG, "extract_regions: null start or end array");
  STB_TRY(use_device(tree));
  Tree& t = const_cast<stb_tree&>(*tree);
  auto d_start = reinterpret_cast<const unsigned long long*>(start), d_end = reinterpret_cast<const unsigned long long*>(end);
  const uint8_t* d_strand = strand;
  if (memory == STB_DEVICE) {
    if ((reinterpret_cast<uintptr_t>(start) | reinterpret_cast<uintptr_t>(end)) & 7u)
      return t.fail(STB_ERR_INVALID_ARG, "extract_regions: start and end must be 8-byte aligned");
  } else {
    const uint64_t words = 8 * n_regions;
    STB_CUDA(t, t.region_inputs.ensure(2 * words + (strand ? n_regions : 0), t.stream));
    char* d = t.region_inputs.ptr;
    Launch l(t, "h2d_copy", false);
    STB_CUDA(t, cudaMemcpyAsync(d, start, words, cudaMemcpyHostToDevice, t.stream));
    STB_CUDA(t, cudaMemcpyAsync(d + words, end, words, cudaMemcpyHostToDevice, t.stream));
    if (strand) STB_CUDA(t, cudaMemcpyAsync(d + 2 * words, strand, n_regions, cudaMemcpyHostToDevice, t.stream));
    d_start = reinterpret_cast<const unsigned long long*>(d);
    d_end = reinterpret_cast<const unsigned long long*>(d + words);
    d_strand = strand ? reinterpret_cast<const uint8_t*>(d + 2 * words) : nullptr;
  }
  RegionPlan plan;
  STB_TRY(region_plan(t, d_start, d_end, d_strand, n_regions, &plan));
  const uint64_t total = plan.total_len;
  *written = total;
  if (!out) return STB_OK;
  if (cap < total) return t.fail(STB_ERR_BUFFER_TOO_SMALL, "extract_regions: cap < total region length");
  if (memory == STB_DEVICE) return region_write(t, d_start, d_end, d_strand, n_regions, plan, out);
  // the output comes back through the handle's grow-only staging buffer
  STB_CUDA(t, t.staging.ensure(total + 16, t.stream));
  STB_TRY(region_write(t, d_start, d_end, d_strand, n_regions, plan, t.staging.ptr));
  return from_device(t, out, t.staging.ptr, total, STB_HOST);
}

const char* stb_status_string(int status) {
  switch (status) {
    case STB_OK: return "ok";
    case STB_ERR_CUDA: return "CUDA error or no CUDA device";
    case STB_ERR_INVALID_ARG: return "invalid argument";
    case STB_ERR_UNKNOWN_SYMBOL: return "unknown nucleotide symbol";
    case STB_ERR_EMPTY: return "input shorter than one leaf";
    case STB_ERR_BUFFER_TOO_SMALL: return "buffer too small";
    case STB_ERR_NOT_BUILT: return "tree not built";
    case STB_ERR_INDEX_CEILING: return "layer exceeds the pointer index range";
    case STB_ERR_BAD_LEAF: return "packed leaf has bits above 4*dna_size";
    case STB_ERR_OUT_OF_RANGE: return "index out of range";
    case STB_ERR_BAD_STREAM: return "malformed .dag stream";
    case STB_ERR_TOO_LARGE: return "input too large";
    default: return "unknown status";
  }
}

const char* stb_last_error(const stb_tree* tree) { return tree ? tree->error.c_str() : ""; }

uint64_t stb_kernel_launches(void) { return stb::g_kernel_launches; }

int stb_profile_enable(stb_tree* tree, int on) {
  if (!tree) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  tree->flush_profile();
  tree->profiling = on != 0;
  return STB_OK;
}

int stb_profile_reset(stb_tree* tree) {
  if (!tree) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  tree->flush_profile();
  tree->acc.clear();
  tree->acc_order.clear();
  return STB_OK;
}

int stb_profile_read(stb_tree* tree, const char** names, double* total_ms, uint64_t* launches, uint64_t cap, uint64_t* count) {
  if (!tree || !count) return STB_ERR_INVALID_ARG;
  STB_TRY(use_device(tree));
  tree->flush_profile();
  *count = tree->acc_order.size();
  for (uint64_t i = 0; i < tree->acc_order.size() && i < cap; ++i) {
    const auto& name = tree->acc_order[i];
    if (names) names[i] = name.c_str();
    if (total_ms) total_ms[i] = tree->acc[name].ms;
    if (launches) launches[i] = tree->acc[name].launches;
  }
  return STB_OK;
}

int stb_synth_genome(int device, void* cuda_stream, char* out_device, uint64_t n_bases, uint64_t first, uint64_t count,
                     uint64_t seed, uint32_t repeat_permille) {
  if (!out_device && count) return STB_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return STB_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return STB_ERR_CUDA;
  Ctx ctx;
  ctx.device = device;
  ctx.stream = (cudaStream_t)cuda_stream;
  return synth_genome(ctx, out_device, n_bases, first, count, seed, repeat_permille);
}

int stb_synth_mask(int device, void* cuda_stream, char* text_device, uint64_t first, uint64_t count, uint64_t seed) {
  if (!text_device && count) return STB_ERR_INVALID_ARG;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return STB_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return STB_ERR_CUDA;
  Ctx ctx;
  ctx.device = device;
  ctx.stream = (cudaStream_t)cuda_stream;
  return synth_mask(ctx, text_device, first, count, seed);
}

}  // extern "C"
