// a1: graph construction on the device.
// Replaces utils.build_graph_from_triplets / comp_deg_norm (reference kgvae/utils.py:127-150) and
// node_norm_to_edge_norm (kgvae/link_predict.py:95-100): reverse-edge doubling, the
// (dst, src, rel) ordering, in-degree normalisation, plus the three edge orderings the message
// passing kernels consume (dst-major, src-major, etype-major), each as 16-byte packed records so a
// kernel needs one 128-bit load per edge.  Sorting is integer work: CUB radix sort (stable).
#include <cub/cub.cuh>
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

// ------------------------------------------------------------------------------------------
// error plumbing shared by all translation units
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int kg_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

extern "C" const char* kg_last_error(void) { return g_err; }
extern "C" int kg_version(void) { return 100; }

int kg_sm_count() {
  static int cached[64] = {0};            // per device: a process may drive several GPUs
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached[dev] = n;
    else
      return 148;
  }
  return cached[dev];
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per device: remember which devices have it for `slot`
bool kg_attr_needed(int slot) {
  static unsigned long long done[8] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || slot < 0 || slot >= 8) return true;
  const unsigned long long bit = 1ull << dev;
  if (done[slot] & bit) return false;
  done[slot] |= bit;
  return true;
}

extern "C" int kg_device_info(int* sm_count, int* cc_major, int* cc_minor) {
  int dev = 0;
  KG_CUDA(cudaGetDevice(&dev));
  KG_CUDA(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev));
  KG_CUDA(cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev));
  KG_CUDA(cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
  return KG_OK;
}

// Peer-visible device buffers (parallel.PeerRows): plain cudaMalloc memory exported with CUDA IPC and
// opened by the other ranks of the node ON THEIR OWN current device with lazy peer access, so that
// their kernels (LDG and the TMA bulk copies alike) can dereference it over NVLink.
extern "C" int kg_peer_alloc(size_t bytes, void** ptr, unsigned char* handle_out /* 64 bytes */) {
  KG_REQUIRE(bytes > 0 && ptr && handle_out, "peer_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  KG_CUDA(cudaMalloc(ptr, bytes));
  KG_CUDA(cudaMemset(*ptr, 0, bytes));
  cudaIpcMemHandle_t h;
  KG_CUDA(cudaIpcGetMemHandle(&h, *ptr));
  memcpy(handle_out, &h, sizeof(h));
  return KG_OK;
}

extern "C" int kg_peer_open(const unsigned char* handle /* 64 bytes */, void** ptr) {
  KG_REQUIRE(handle && ptr, "peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  KG_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return KG_OK;
}

extern "C" int kg_peer_close(void* ptr) {
  KG_CUDA(cudaIpcCloseMemHandle(ptr));
  return KG_OK;
}

extern "C" int kg_peer_free(void* ptr) {
  KG_CUDA(cudaFree(ptr));
  return KG_OK;
}

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
static constexpr int kThreads = 256;

// key = dst:24 | src:24 | rel:16  -> ascending key order == ascending (dst, src, rel)
__global__ void make_edge_keys(const int* __restrict__ src, const int* __restrict__ rel,
                               const int* __restrict__ dst, int T, int R, unsigned long long* keys) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  unsigned long long s = (unsigned)src[i], d = (unsigned)dst[i], r = (unsigned)rel[i];
  keys[i] = (d << 40) | (s << 16) | r;                // s -> d with rel
  keys[T + i] = (s << 40) | (d << 16) | (r + R);      // d -> s with rel + R
}

__global__ void decode_edge_keys(const unsigned long long* __restrict__ keys, int E, int* e_src,
                                 int* e_dst, int* e_type) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= E) return;
  unsigned long long k = keys[i];
  e_dst[i] = (int)(k >> 40);
  e_src[i] = (int)((k >> 16) & 0xffffffull);
  e_type[i] = (int)(k & 0xffffull);
}

// The relation histogram has few bins (474 at the FB15k-237 shape) and real relation frequencies are heavy-tailed:
// one global atomic per edge serialises on the popular relations' counters.  With R2 <= kRelSmemBins the CTA counts
// its edges in shared memory and adds each non-empty bin once.
constexpr int kRelSmemBins = 4096;

__global__ void histogram3(const int* __restrict__ e_src, const int* __restrict__ e_dst,
                           const int* __restrict__ e_type, int E, int R2, int* deg_in, int* deg_out,
                           int* cnt_rel) {
  extern __shared__ int rel_s[];
  const bool local = R2 <= kRelSmemBins;
  if (local) {
    for (int b = threadIdx.x; b < R2; b += blockDim.x) rel_s[b] = 0;
    __syncthreads();
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < E; i += gridDim.x * blockDim.x) {
    atomicAdd(&deg_in[e_dst[i]], 1);
    atomicAdd(&deg_out[e_src[i]], 1);
    if (local) atomicAdd(&rel_s[e_type[i]], 1);
    else atomicAdd(&cnt_rel[e_type[i]], 1);
  }
  if (local) {
    __syncthreads();
    for (int b = threadIdx.x; b < R2; b += blockDim.x)
      if (rel_s[b]) atomicAdd(&cnt_rel[b], rel_s[b]);
  }
}

// norm_v = 1/in_deg(v), inf -> 0 (kgvae/utils.py:127-132); float division, round-to-nearest
__global__ void degree_norm(const int* __restrict__ row_ptr, int N, float* norm) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= N) return;
  int d = row_ptr[v + 1] - row_ptr[v];
  norm[v] = d > 0 ? 1.0f / (float)d : 0.0f;
}

__global__ void iota(int* x, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = i;
}

// which: 0 dst-major {src, etype, norm, dst}; 1 src-major {dst, etype, norm, edge};
//        2 etype-major {src, dst, etype, norm}
__global__ void fill_pack(const int* __restrict__ perm, const int* __restrict__ e_src,
                          const int* __restrict__ e_dst, const int* __restrict__ e_type,
                          const float* __restrict__ e_norm, const float* __restrict__ node_norm,
                          int E, int which, int4* pack) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= E) return;
  int e = perm ? perm[k] : k;
  int s = e_src[e], d = e_dst[e], t = e_type[e];
  float nv = e_norm ? e_norm[e] : (node_norm ? node_norm[d] : 1.0f);
  int nb = __float_as_int(nv);
  int4 p;
  if (which == 0) p = make_int4(s, t, nb, d);
  else if (which == 1) p = make_int4(d, t, nb, e);
  else p = make_int4(s, d, t, nb);
  pack[k] = p;
}

static int bits_for(int n) {
  int b = 1;
  while (b < 31 && (1ll << b) < (long long)n) ++b;
  return b;
}

// ------------------------------------------------------------------------------------------
// index building shared by both entry points
// ------------------------------------------------------------------------------------------
static size_t cub_temp_bytes(int E, int N, int R) {
  size_t a = 0, b = 0, c = 0;
  cub::DeviceRadixSort::SortKeys((void*)nullptr, a, (unsigned long long*)nullptr,
                                 (unsigned long long*)nullptr, E);
  cub::DeviceRadixSort::SortPairs((void*)nullptr, b, (int*)nullptr, (int*)nullptr, (int*)nullptr,
                                  (int*)nullptr, E);
  int m = (N > R ? N : R) + 1;
  cub::DeviceScan::ExclusiveSum((void*)nullptr, c, (int*)nullptr, (int*)nullptr, m);
  size_t t = a > b ? a : b;
  return kg_align_up((t > c ? t : c) + 256);
}

static size_t index_workspace(int E) {
  // 4 int arrays of E (keys in/out, vals in/out) + cub temp (sized for E; N, R <= 2^24 bounded below)
  return 4 * kg_align_up((size_t)E * 4) + cub_temp_bytes(E, 1 << 24, 1 << 16) + 1024;
}

static int build_index(const int* e_src, const int* e_dst, const int* e_type, const float* e_norm,
                       const float* node_norm, int E, int N, int R2, int* row_ptr, int4* fwd_pack,
                       int* col_ptr, int4* bwd_pack, int* rel_ptr, int4* rel_pack, KgArena& ws,
                       bool dst_sorted, cudaStream_t st) {
  int* keys_in = ws.take<int>(E);
  int* keys_out = ws.take<int>(E);
  int* vals_in = ws.take<int>(E);
  int* vals_out = ws.take<int>(E);
  size_t temp_bytes = cub_temp_bytes(E, N, R2);
  void* temp = ws.take<char>(temp_bytes);
  if (!keys_in || !keys_out || !vals_in || !vals_out || !temp)
    return kg_fail(KG_ERR_WORKSPACE, "graph index: workspace too small");
  const int gridE = kg_div_up(E, kThreads);

  KG_CUDA(cudaMemsetAsync(row_ptr, 0, sizeof(int) * (N + 1), st));
  KG_CUDA(cudaMemsetAsync(col_ptr, 0, sizeof(int) * (N + 1), st));
  KG_CUDA(cudaMemsetAsync(rel_ptr, 0, sizeof(int) * (R2 + 1), st));
  if (E > 0) {
    const int grid_h = gridE < 8 * kg_sm_count() ? gridE : 8 * kg_sm_count();   // full occupancy; a popular relation's counter: <= grid_h adds
    histogram3<<<grid_h, kThreads, R2 <= kRelSmemBins ? sizeof(int) * R2 : 0, st>>>(e_src, e_dst, e_type, E, R2, row_ptr,
                                                                                     col_ptr, rel_ptr);
    KG_LAUNCH_OK();
  }
  size_t tb = temp_bytes;
  KG_CUDA(cub::DeviceScan::ExclusiveSum(temp, tb, row_ptr, row_ptr, N + 1, st));
  tb = temp_bytes;
  KG_CUDA(cub::DeviceScan::ExclusiveSum(temp, tb, col_ptr, col_ptr, N + 1, st));
  tb = temp_bytes;
  KG_CUDA(cub::DeviceScan::ExclusiveSum(temp, tb, rel_ptr, rel_ptr, R2 + 1, st));
  if (E == 0) return KG_OK;

  iota<<<gridE, kThreads, 0, st>>>(vals_in, E);
  KG_LAUNCH_OK();
  // dst-major (stable: original order is the tie-break); optional
  if (fwd_pack == nullptr) {
  } else if (dst_sorted) {
    fill_pack<<<gridE, kThreads, 0, st>>>(nullptr, e_src, e_dst, e_type, e_norm, node_norm, E, 0, fwd_pack);
  } else {
    tb = temp_bytes;
    KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, tb, e_dst, keys_out, vals_in, vals_out, E, 0,
                                            bits_for(N), st));
    fill_pack<<<gridE, kThreads, 0, st>>>(vals_out, e_src, e_dst, e_type, e_norm, node_norm, E, 0, fwd_pack);
  }
  KG_LAUNCH_OK();
  // src-major; optional
  if (bwd_pack != nullptr) {
    tb = temp_bytes;
    KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, tb, e_src, keys_out, vals_in, vals_out, E, 0,
                                            bits_for(N), st));
    fill_pack<<<gridE, kThreads, 0, st>>>(vals_out, e_src, e_dst, e_type, e_norm, node_norm, E, 1, bwd_pack);
    KG_LAUNCH_OK();
  }
  // etype-major
  tb = temp_bytes;
  KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, tb, e_type, keys_out, vals_in, vals_out, E, 0,
                                          bits_for(R2), st));
  fill_pack<<<gridE, kThreads, 0, st>>>(vals_out, e_src, e_dst, e_type, e_norm, node_norm, E, 2, rel_pack);
  KG_LAUNCH_OK();
  (void)keys_in;
  return KG_OK;
}

extern "C" size_t kg_graph_index_workspace_bytes(int n_edges) {
  return index_workspace(n_edges > 0 ? n_edges : 1);
}

extern "C" int kg_graph_index(const int32_t* e_src, const int32_t* e_dst, const int32_t* e_type,
                              const float* e_norm, int n_edges, int num_nodes, int num_etypes,
                              int32_t* row_ptr, void* fwd_pack, int32_t* col_ptr, void* bwd_pack,
                              int32_t* rel_ptr, void* rel_pack, void* workspace,
                              size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_edges >= 0 && num_nodes > 0 && num_etypes > 0, "graph_index: bad sizes");
  KG_REQUIRE(num_nodes < (1 << 24) && num_etypes < (1 << 16), "graph_index: N < 2^24, R < 2^16");
  KgArena ws(workspace, workspace_bytes);
  return build_index(e_src, e_dst, e_type, e_norm, nullptr, n_edges, num_nodes, num_etypes, row_ptr,
                     (int4*)fwd_pack, col_ptr, (int4*)bwd_pack, rel_ptr, (int4*)rel_pack, ws, false,
                     kg_stream(stream));
}

// ------------------------------------------------------------------------------------------
// node-tiled relation-major list (graphs whose feature matrices exceed L2)
// ------------------------------------------------------------------------------------------
__global__ void tiled_rel_keys(const int* __restrict__ e_node, const int* __restrict__ e_type, int E,
                               int tile_nodes, int type_bits, unsigned* keys) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= E) return;
  keys[i] = ((unsigned)(e_node[i] / tile_nodes) << type_bits) | (unsigned)e_type[i];
}

extern "C" size_t kg_graph_rel_tiled_workspace_bytes(int n_edges) {
  int E = n_edges > 0 ? n_edges : 1;
  size_t a = 0;
  cub::DeviceRadixSort::SortPairs((void*)nullptr, a, (unsigned*)nullptr, (unsigned*)nullptr, (int*)nullptr,
                                  (int*)nullptr, E);
  return 4 * kg_align_up((size_t)E * 4) + kg_align_up(a + 256) + 1024;
}

extern "C" int kg_graph_rel_tiled(const int32_t* e_src, const int32_t* e_dst, const int32_t* e_type,
                                  const float* e_norm, int n_edges, int num_nodes, int num_etypes,
                                  int tile_nodes, int by_src, void* pack_out, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_edges >= 0 && num_nodes > 0 && num_etypes > 0 && tile_nodes > 0, "graph_rel_tiled: bad sizes");
  const int E = n_edges;
  if (E == 0) return KG_OK;
  const int tiles = (num_nodes + tile_nodes - 1) / tile_nodes;
  const int type_bits = bits_for(num_etypes), tile_bits = bits_for(tiles);
  KG_REQUIRE(type_bits + tile_bits <= 32, "graph_rel_tiled: tile and relation ids exceed a 32-bit key");
  cudaStream_t st = kg_stream(stream);
  KgArena ws(workspace, workspace_bytes);
  unsigned* k_in = ws.take<unsigned>(E);
  unsigned* k_out = ws.take<unsigned>(E);
  int* v_in = ws.take<int>(E);
  int* v_out = ws.take<int>(E);
  size_t temp_bytes = 0;
  cub::DeviceRadixSort::SortPairs((void*)nullptr, temp_bytes, k_in, k_out, v_in, v_out, E);
  void* temp = ws.take<char>(temp_bytes + 256);
  if (!k_in || !k_out || !v_in || !v_out || !temp)
    return kg_fail(KG_ERR_WORKSPACE, "graph_rel_tiled: workspace too small");
  const int gridE = kg_div_up(E, kThreads);
  tiled_rel_keys<<<gridE, kThreads, 0, st>>>(by_src ? e_src : e_dst, e_type, E, tile_nodes, type_bits, k_in);
  KG_LAUNCH_OK();
  iota<<<gridE, kThreads, 0, st>>>(v_in, E);
  KG_LAUNCH_OK();
  KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, temp_bytes, k_in, k_out, v_in, v_out, E, 0, type_bits + tile_bits,
                                          st));
  fill_pack<<<gridE, kThreads, 0, st>>>(v_out, e_src, e_dst, e_type, e_norm, nullptr, E, 2,
                                        reinterpret_cast<int4*>(pack_out));
  KG_LAUNCH_OK();
  return KG_OK;
}

__global__ void patch_pack_norm(int4* fwd, int4* bwd, int4* rel, const float* node_norm, int E) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= E) return;
  if (fwd) {
    int4 f = fwd[k];
    f.z = __float_as_int(node_norm[f.w]);      // {src, etype, norm, dst}
    fwd[k] = f;
  }
  if (bwd) {
    int4 b = bwd[k];
    b.z = __float_as_int(node_norm[b.x]);      // {dst, etype, norm, edge}
    bwd[k] = b;
  }
  int4 r = rel[k];
  r.w = __float_as_int(node_norm[r.y]);      // {src, dst, etype, norm}
  rel[k] = r;
}

extern "C" size_t kg_graph_build_workspace_bytes(int n_triplets) {
  int E = 2 * (n_triplets > 0 ? n_triplets : 1);
  return 2 * kg_align_up((size_t)E * 8) + index_workspace(E) + 1024;
}

extern "C" int kg_graph_build(const int32_t* src, const int32_t* rel, const int32_t* dst,
                              int n_triplets, int num_nodes, int num_rels, int32_t* e_src,
                              int32_t* e_dst, int32_t* e_type, int32_t* row_ptr, float* node_norm,
                              void* fwd_pack, int32_t* col_ptr, void* bwd_pack, int32_t* rel_ptr,
                              void* rel_pack, void* workspace, size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_triplets >= 0 && num_nodes > 0 && num_rels > 0, "graph_build: bad sizes");
  KG_REQUIRE(num_nodes < (1 << 24) && 2 * num_rels < (1 << 16), "graph_build: N < 2^24, 2R < 2^16");
  cudaStream_t st = kg_stream(stream);
  const int T = n_triplets, E = 2 * T, R2 = 2 * num_rels;
  KgArena ws(workspace, workspace_bytes);
  unsigned long long* k_in = ws.take<unsigned long long>(E > 0 ? E : 1);
  unsigned long long* k_out = ws.take<unsigned long long>(E > 0 ? E : 1);
  if (!k_in || !k_out) return kg_fail(KG_ERR_WORKSPACE, "graph_build: workspace too small");
  if (E > 0) {
    make_edge_keys<<<kg_div_up(T, kThreads), kThreads, 0, st>>>(src, rel, dst, T, num_rels, k_in);
    KG_LAUNCH_OK();
    // reuse the index arena's cub temp for the 64-bit sort: take it, then rewind
    size_t mark = ws.used;
    size_t temp_bytes = cub_temp_bytes(E, num_nodes, R2);
    void* temp = ws.take<char>(temp_bytes);
    if (!temp) return kg_fail(KG_ERR_WORKSPACE, "graph_build: workspace too small");
    KG_CUDA(cub::DeviceRadixSort::SortKeys(temp, temp_bytes, k_in, k_out, E, 0,
                                           40 + bits_for(num_nodes), st));
    ws.used = mark;
    decode_edge_keys<<<kg_div_up(E, kThreads), kThreads, 0, st>>>(k_out, E, e_src, e_dst, e_type);
    KG_LAUNCH_OK();
  }
  // CSR first (norm needs in-degrees), then packs with norm[dst]
  // build_index computes row_ptr; node_norm is derived between histogram and pack filling, so the
  // packs are filled by a second pass below once node_norm exists.
  int rc = build_index(e_src, e_dst, e_type, nullptr, nullptr, E, num_nodes, R2, row_ptr,
                       (int4*)fwd_pack, col_ptr, (int4*)bwd_pack, rel_ptr, (int4*)rel_pack, ws, true, st);
  if (rc != KG_OK) return rc;
  degree_norm<<<kg_div_up(num_nodes, kThreads), kThreads, 0, st>>>(row_ptr, num_nodes, node_norm);
  KG_LAUNCH_OK();
  if (E > 0) {
    // rewrite the norm field of every record now that node_norm is known
    patch_pack_norm<<<kg_div_up(E, kThreads), kThreads, 0, st>>>((int4*)fwd_pack, (int4*)bwd_pack,
                                                               (int4*)rel_pack, node_norm, E);
    KG_LAUNCH_OK();
  }
  return KG_OK;
}

// ------------------------------------------------------------------------------------------
// relabelling of a sampled edge set with a fixed node budget (utils.SampledDeviceSampler)
// np.unique((src, dst), return_inverse=True) of kgvae/utils.py:85-124, with every size fixed by B and cap so the
// call can sit inside a CUDA-graph capture: the 2B endpoint ids are sorted with their slots, a head flag marks
// the first of each run of equal ids, an inclusive scan of the flags numbers the runs, and one scatter writes
// the labels back to the slots and each distinct id to node_id[label].  Rows n_valid .. cap-1 of node_id are
// padding: row i looks up entity i (an id in range that is used at most once more, so the embedding backward's
// per-element atomics never pile up on one row).
// ------------------------------------------------------------------------------------------
__global__ void relabel_keys(const int* __restrict__ picked, int B, int* __restrict__ keys, int* __restrict__ slots,
                             int* __restrict__ rel) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  keys[i] = picked[3 * i];
  keys[B + i] = picked[3 * i + 2];
  slots[i] = i;
  slots[B + i] = B + i;
  rel[i] = picked[3 * i + 1];
}

__global__ void relabel_heads(const int* __restrict__ sorted, int M, int* __restrict__ flags) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  flags[i] = (i == 0 || sorted[i] != sorted[i - 1]) ? 1 : 0;
}

__global__ void relabel_scatter(const int* __restrict__ sorted, const int* __restrict__ slots,
                                const int* __restrict__ run, int B, int cap, int* __restrict__ node_id,
                                int* __restrict__ src, int* __restrict__ dst, int* __restrict__ n_valid) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int M = 2 * B;
  const int nv = run[M - 1];                          // number of distinct ids
  if (i < M) {
    const int label = run[i] - 1;
    const int s = slots[i];
    if (s < B) src[s] = label;
    else dst[s - B] = label;
    if ((i == 0 || sorted[i] != sorted[i - 1]) && label < cap) node_id[label] = sorted[i];
  }
  if (i < cap && i >= nv) node_id[i] = i;             // padding row i looks up entity i
  // a caller that breaks cap >= distinct ids still gets n_valid <= cap: nothing drawn from [0, n_valid) can index past
  // the node set (the ids past cap are dropped, their labels are not meaningful)
  if (i == 0) n_valid[0] = nv < cap ? nv : cap;
}

static size_t relabel_cub_bytes(int M) {
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortPairs((void*)nullptr, a, (int*)nullptr, (int*)nullptr, (int*)nullptr, (int*)nullptr, M);
  cub::DeviceScan::InclusiveSum((void*)nullptr, b, (int*)nullptr, (int*)nullptr, M);
  return kg_align_up((a > b ? a : b) + 256);
}

extern "C" size_t kg_sample_relabel_workspace_bytes(int n_picks) {
  const int M = 2 * (n_picks > 0 ? n_picks : 1);
  return 5 * kg_align_up((size_t)M * 4) + relabel_cub_bytes(M) + 1024;
}

extern "C" int kg_sample_relabel(const int32_t* picked, int n_picks, int num_nodes, int cap, int32_t* node_id,
                                 int32_t* src, int32_t* rel, int32_t* dst, int32_t* n_valid, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_picks > 0 && num_nodes > 0 && n_picks < (1 << 29), "sample_relabel: bad sizes");
  KG_REQUIRE(cap > 0 && cap <= num_nodes && cap <= 2 * n_picks, "sample_relabel: need 0 < cap <= min(2B, num_nodes)");
  cudaStream_t st = kg_stream(stream);
  const int B = n_picks, M = 2 * B;
  KgArena ws(workspace, workspace_bytes);
  int* k_in = ws.take<int>(M);
  int* k_out = ws.take<int>(M);
  int* s_in = ws.take<int>(M);
  int* s_out = ws.take<int>(M);
  int* run = ws.take<int>(M);
  size_t temp_bytes = relabel_cub_bytes(M);
  void* temp = ws.take<char>(temp_bytes);
  if (!k_in || !k_out || !s_in || !s_out || !run || !temp)
    return kg_fail(KG_ERR_WORKSPACE, "sample_relabel: workspace too small");
  relabel_keys<<<kg_div_up(B, kThreads), kThreads, 0, st>>>(picked, B, k_in, s_in, rel);
  KG_LAUNCH_OK();
  size_t tb = temp_bytes;
  KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, tb, k_in, k_out, s_in, s_out, M, 0, bits_for(num_nodes), st));
  relabel_heads<<<kg_div_up(M, kThreads), kThreads, 0, st>>>(k_out, M, run);
  KG_LAUNCH_OK();
  tb = temp_bytes;
  KG_CUDA(cub::DeviceScan::InclusiveSum(temp, tb, run, run, M, st));
  relabel_scatter<<<kg_div_up(M > cap ? M : cap, kThreads), kThreads, 0, st>>>(k_out, s_out, run, B, cap, node_id, src,
                                                                               dst, n_valid);
  KG_LAUNCH_OK();
  return KG_OK;
}

