// a9: DistMult decoder, BCE-with-logits and the L2 regulariser, forward and backward.
// Replaces LinkPredict.calc_score / get_loss / regularization_loss (reference
// kgvae/link_predict.py:57-78).  The reference gathers three [S, h] tensors, materialises two
// [S, h] products and, in backward, scatter-adds with index_put(accumulate) into z.
// Here: the score is one warp-level pass over three gathered rows; the backward into z is a
// gather-reduce over an entity-major index of the triplets (no atomics, deterministic), the
// backward into w_relation runs over relation-grouped triplets.
#include <cub/cub.cuh>

#include "common.cuh"

static constexpr int kThreads = 256;

// ------------------------------------------------------------------------------------------
// score_i = sum_d z[s,d] w[r,d] z[o,d] + shift          (link_predict.py:57-63, :75-76)
// ------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(kThreads)
distmult_score_kernel(const float* __restrict__ z, const float* __restrict__ w,
                      const int* __restrict__ trip, int S, int h, const float* __restrict__ shift,
                      float* __restrict__ score) {
  const int t = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= S) return;
  const int s = __ldg(trip + 3 * (size_t)t), r = __ldg(trip + 3 * (size_t)t + 1),
            o = __ldg(trip + 3 * (size_t)t + 2);
  float acc = 0.f;
  if (VEC == 4) {
    const float4* zs = reinterpret_cast<const float4*>(z + (size_t)s * h);
    const float4* wr = reinterpret_cast<const float4*>(w + (size_t)r * h);
    const float4* zo = reinterpret_cast<const float4*>(z + (size_t)o * h);
    for (int c = lane; c < h / 4; c += 32) {
      const float4 a = __ldg(zs + c), b = __ldg(wr + c), d = __ldg(zo + c);
      acc = fmaf(a.x * b.x, d.x, acc);
      acc = fmaf(a.y * b.y, d.y, acc);
      acc = fmaf(a.z * b.z, d.z, acc);
      acc = fmaf(a.w * b.w, d.w, acc);
    }
  } else {
    for (int c = lane; c < h; c += 32)
      acc = fmaf(__ldg(z + (size_t)s * h + c) * __ldg(w + (size_t)r * h + c), __ldg(z + (size_t)o * h + c), acc);
  }
  acc = kg_warp_sum(acc);
  if (lane == 0) score[t] = shift ? acc + __ldg(shift) : acc;
}

extern "C" int kg_distmult_score(const float* z, const float* w, const int32_t* triplets,
                                 int n_triplets, int h, const float* shift, float* score, void* stream) {
  KG_REQUIRE(n_triplets >= 0 && h > 0, "distmult score: bad sizes");
  if (n_triplets == 0) return KG_OK;
  const int grid = kg_div_up((long long)n_triplets * 32, kThreads);
  const bool vec = (h % 4 == 0) && ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(w)) & 15) == 0;
  if (vec) distmult_score_kernel<4><<<grid, kThreads, 0, kg_stream(stream)>>>(z, w, triplets, n_triplets, h, shift, score);
  else distmult_score_kernel<1><<<grid, kThreads, 0, kg_stream(stream)>>>(z, w, triplets, n_triplets, h, shift, score);
  KG_LAUNCH_OK();
  return KG_OK;
}

// ------------------------------------------------------------------------------------------
// deterministic two-stage reductions
// ------------------------------------------------------------------------------------------
static constexpr int kMaxPartials = 1024;

static int reduce_blocks(long long n) {
  long long b = (n + 4 * kThreads - 1) / (4 * kThreads);
  return (int)(b < 1 ? 1 : (b > kMaxPartials ? kMaxPartials : b));
}

__device__ __forceinline__ float block_sum(float v) {
  __shared__ float red[kThreads / 32];
  v = kg_warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float tot = 0.f;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) tot += red[i];
  }
  return tot;   // valid on thread 0
}

// mode 0: sum x; 1: sum x^2; 2: BCE-with-logits(x, y) and dscore = (sigmoid(x) - y) * inv_n
__global__ void __launch_bounds__(kThreads)
reduce_stage1(const float* __restrict__ x, const float* __restrict__ y, long long n, int mode,
              float inv_n, float* __restrict__ dscore, float* __restrict__ partial,
              const int* __restrict__ n_rows = nullptr, int row_len = 0) {
  // n_rows (device, may be NULL): only the first n_rows rows of row_len elements are read
  if (n_rows != nullptr) n = min(n, (long long)__ldg(n_rows) * row_len);
  float s = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float v = x[i];
    if (mode == 0) s += v;
    else if (mode == 1) s = fmaf(v, v, s);
    else {
      const float lab = y[i];
      s += fmaxf(v, 0.f) - v * lab + log1pf(expf(-fabsf(v)));   // F.binary_cross_entropy_with_logits
      if (dscore) dscore[i] = (kg_sigmoid(v) - lab) * inv_n;
    }
  }
  const float tot = block_sum(s);
  if (threadIdx.x == 0) partial[blockIdx.x] = tot;
}

__global__ void reduce_stage2(const float* __restrict__ partial, int count, float scale,
                              float* __restrict__ out) {
  // one warp, fixed order: lane-strided partial sums then a shuffle tree
  float s = 0.f;
  for (int i = threadIdx.x; i < count; i += 32) s += partial[i];
  s = kg_warp_sum(s);
  if (threadIdx.x == 0) out[0] = s * scale;
}

extern "C" size_t kg_reduce_workspace_bytes(long long n) {
  (void)n;
  return kg_align_up(sizeof(float) * kMaxPartials);
}

static int run_reduce(const float* x, const float* y, long long n, int mode, float scale, float inv_n,
                      float* dscore, float* out, void* workspace, size_t workspace_bytes, cudaStream_t st,
                      const int* n_rows = nullptr, int row_len = 0) {
  if (workspace_bytes < sizeof(float) * kMaxPartials)
    return kg_fail(KG_ERR_WORKSPACE, "reduce: workspace too small");
  if (n == 0) {
    KG_CUDA(cudaMemsetAsync(out, 0, sizeof(float), st));
    return KG_OK;
  }
  const int blocks = reduce_blocks(n);
  float* partial = reinterpret_cast<float*>(workspace);
  reduce_stage1<<<blocks, kThreads, 0, st>>>(x, y, n, mode, inv_n, dscore, partial, n_rows, row_len);
  KG_LAUNCH_OK();
  reduce_stage2<<<1, 32, 0, st>>>(partial, blocks, scale, out);
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" int kg_bce_logits_fwd(const float* score, const float* labels, int n, float* loss_out,
                                 float* dscore, void* workspace, size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n >= 0, "bce: bad size");
  const float inv = n > 0 ? 1.0f / (float)n : 0.f;
  return run_reduce(score, labels, n, 2, inv, inv, dscore, loss_out, workspace, workspace_bytes, kg_stream(stream));
}

extern "C" int kg_sum_squares(const float* x, long long n, float* out, void* workspace,
                              size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n >= 0, "sum_squares: bad size");
  return run_reduce(x, nullptr, n, 1, 1.f, 0.f, nullptr, out, workspace, workspace_bytes, kg_stream(stream));
}

// sum of squares over the first n_valid (device int) rows of an [n_rows, h] matrix: the regulariser mean(z^2) of a
// sampled subgraph padded to a fixed node budget (the grid is sized by n_rows; no host read of n_valid)
extern "C" int kg_sum_squares_rows(const float* x, int n_rows, int h, const int32_t* n_valid, float* out,
                                   void* workspace, size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_rows >= 0 && h > 0 && n_valid != nullptr, "sum_squares_rows: bad arguments");
  return run_reduce(x, nullptr, (long long)n_rows * h, 1, 1.f, 0.f, nullptr, out, workspace, workspace_bytes,
                    kg_stream(stream), n_valid, h);
}

extern "C" int kg_sum(const float* x, long long n, float* out, void* workspace, size_t workspace_bytes,
                      void* stream) {
  KG_REQUIRE(n >= 0, "sum: bad size");
  return run_reduce(x, nullptr, n, 0, 1.f, 0.f, nullptr, out, workspace, workspace_bytes, kg_stream(stream));
}

// ------------------------------------------------------------------------------------------
// triplet index: the two orderings the decoder kernels walk (integer work: CUB radix sort, no atomics)
//   rs_rec  [S]  int4 {s, r, o, t}        sorted by (r, s): runs share w[r] and z[s]
//   ent_ptr [n_nodes+1], ent_pack [2S] int4 {other, r, t, 0} sorted by (entity, r): for entity v every
//           triplet where v is subject (other = object) or object (other = subject)
// ------------------------------------------------------------------------------------------
// DistMult is symmetric in its two entities (score = sum_d z[s,d] w[r,d] z[o,d]), so a triplet may be
// walked from either end.  The (r, a)-ordered pass keeps z[a] and dz[a] in registers over a run of
// equal (r, a), so the end with the LONGER run should lead: with negative sampling a positive and the
// negatives that corrupt its other end share it (runs of ~6 instead of 1).  Run lengths are estimated
// with a hashed counter table - collisions only cost speed, never correctness.
// Table size: 2^22 counters up to 4 M triplets (the FB15k-237 step: 3 M); beyond that about two slots per triplet,
// at most 2^28 (1 GB) - at the ogbl-wikikg2 shape (176 M triplets, 32 M distinct (relation, entity) pairs) a 4 M-slot
// table made every count a sum over ~8 unrelated pairs, the orientation came out random and the runs 1.8 triplets
// long instead of ~5.5 (ncu: 5 KB of DRAM reads per triplet instead of 3 KB).
static int orient_bits(int S) {
  if (S <= (1 << 22)) return 22;
  int b = 23;
  while (b < 28 && (1LL << b) < 2LL * S) ++b;
  return b;
}

__device__ __forceinline__ unsigned orient_slot(unsigned r, unsigned e, unsigned mask) {
  unsigned x = r * 0x9E3779B1u ^ (e + 0x7F4A7C15u) * 0x85EBCA6Bu;
  x ^= x >> 15;
  x *= 0x2C1B3C6Du;
  x ^= x >> 13;
  return x & mask;
}

__global__ void orient_count(const int* __restrict__ trip, int S, unsigned* __restrict__ table, unsigned mask) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= S) return;
  const unsigned s = (unsigned)trip[3 * (size_t)t], r = (unsigned)trip[3 * (size_t)t + 1],
                 o = (unsigned)trip[3 * (size_t)t + 2];
  atomicAdd(table + orient_slot(r, s, mask), 1u);
  atomicAdd(table + orient_slot(r, o, mask), 1u);
}

// rs_key leads with whichever end has the longer (estimated) run; bit 31 of rs_val marks a swap.
// KeyT: 32-bit keys when relation and entity bits fit (23 bits at the FB15k-237 shape) - a third less sort traffic.
// ent_mode 1: (entity, r) keys for BOTH ends of every triplet (2S entries); 2: for the TRAILING end only - the one
// the (r, leading entity)-ordered pass does not keep in registers (S entries; bit 31 of ent_val marks a swap)
template <typename KeyT>
__global__ void triplet_keys(const int* __restrict__ trip, int S, int nb, int rb,
                             const unsigned* __restrict__ table, KeyT* rs_key, int* rs_val,
                             KeyT* ent_key, int* ent_val, int ent_mode, unsigned mask) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= S) return;
  const KeyT s = (unsigned)trip[3 * (size_t)t], r = (unsigned)trip[3 * (size_t)t + 1],
             o = (unsigned)trip[3 * (size_t)t + 2];
  const bool swap = table != nullptr && table[orient_slot((unsigned)r, (unsigned)o, mask)] > table[orient_slot((unsigned)r, (unsigned)s, mask)];
  rs_key[t] = (r << nb) | (swap ? o : s);
  rs_val[t] = swap ? (t | 0x80000000) : t;
  if (ent_key && ent_mode == 2) {
    ent_key[t] = ((swap ? s : o) << rb) | r;
    ent_val[t] = swap ? (t | 0x80000000) : t;
  } else if (ent_key) {
    ent_key[t] = (s << rb) | r;      ent_val[t] = t;          // subject side
    ent_key[S + t] = (o << rb) | r;  ent_val[S + t] = S + t;  // object side
  }
}

// rec = {leading entity, relation, other entity, triplet}
__global__ void fill_rs_rec(const int* __restrict__ trip, const int* __restrict__ sorted_val, int S,
                            int4* __restrict__ rec) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= S) return;
  const int v = sorted_val[k], t = v & 0x7fffffff;
  const int s = trip[3 * (size_t)t], o = trip[3 * (size_t)t + 2];
  rec[k] = v < 0 ? make_int4(o, trip[3 * (size_t)t + 1], s, t) : make_int4(s, trip[3 * (size_t)t + 1], o, t);
}

__global__ void fill_ent_pack(const int* __restrict__ trip, const int* __restrict__ sorted_val, int S,
                              int4* __restrict__ pack) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= 2 * S) return;
  const int v = sorted_val[k];
  const int t = v < S ? v : v - S;
  const int other = v < S ? trip[3 * (size_t)t + 2] : trip[3 * (size_t)t];
  pack[k] = make_int4(other, trip[3 * (size_t)t + 1], t, 0);
}

// trailing-end index: pack = {leading entity, relation, triplet, 0}
__global__ void fill_trail_pack(const int* __restrict__ trip, const int* __restrict__ sorted_val, int S,
                                int4* __restrict__ pack) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= S) return;
  const int v = sorted_val[k], t = v & 0x7fffffff;
  pack[k] = make_int4(v < 0 ? trip[3 * (size_t)t + 2] : trip[3 * (size_t)t], trip[3 * (size_t)t + 1], t, 0);
}

// ptr[v] = first position whose key has entity >= v (keys sorted ascending)
template <typename KeyT>
__global__ void ent_lower_bound(const KeyT* __restrict__ keys, int n, int rb, int n_nodes,
                                int* __restrict__ ptr) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v > n_nodes) return;
  if (v == n_nodes) { ptr[v] = n; return; }          // (v << rb) may not fit a 32-bit key for v = n_nodes
  const KeyT want = (KeyT)v << rb;
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(keys + mid) < want) lo = mid + 1;
    else hi = mid;
  }
  ptr[v] = lo;
}

static int bits_for(int n) {
  int b = 1;
  while (b < 31 && (1ll << b) < (long long)n) ++b;
  return b;
}

static size_t triplet_cub_bytes(int S) {
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortPairs((void*)nullptr, a, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                  (int*)nullptr, (int*)nullptr, 2 * S);
  cub::DeviceRadixSort::SortPairs((void*)nullptr, b, (unsigned*)nullptr, (unsigned*)nullptr, (int*)nullptr,
                                  (int*)nullptr, 2 * S);
  return kg_align_up((a > b ? a : b) + 256);
}

template <typename KeyT>
static int triplet_sorts(const int32_t* triplets, int S, int n_nodes, int nb, int rb, const unsigned* table, unsigned mask, int ent_mode,
                         KeyT* rk_in, KeyT* rk_out, int* rv_in, int* rv_out, KeyT* ek_in, KeyT* ek_out, int* ev_in,
                         int* ev_out, void* temp, size_t temp_bytes, void* rs_rec, int32_t* ent_ptr, void* ent_pack,
                         cudaStream_t st) {
  triplet_keys<KeyT><<<kg_div_up(S, kThreads), kThreads, 0, st>>>(triplets, S, nb, rb, table, rk_in, rv_in,
                                                                  ent_mode ? ek_in : nullptr, ev_in, ent_mode, mask);
  KG_LAUNCH_OK();
  size_t tb = temp_bytes;
  if (ent_mode) {
    const int n_ent = ent_mode == 2 ? S : 2 * S;
    KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, tb, ek_in, ek_out, ev_in, ev_out, n_ent, 0, nb + rb, st));
    if (ent_mode == 2) fill_trail_pack<<<kg_div_up(S, kThreads), kThreads, 0, st>>>(triplets, ev_out, S, reinterpret_cast<int4*>(ent_pack));
    else fill_ent_pack<<<kg_div_up(2LL * S, kThreads), kThreads, 0, st>>>(triplets, ev_out, S, reinterpret_cast<int4*>(ent_pack));
    KG_LAUNCH_OK();
    ent_lower_bound<KeyT><<<kg_div_up(n_nodes + 1, kThreads), kThreads, 0, st>>>(ek_out, n_ent, rb, n_nodes, ent_ptr);
    KG_LAUNCH_OK();
  }
  tb = temp_bytes;
  KG_CUDA(cub::DeviceRadixSort::SortPairs(temp, tb, rk_in, rk_out, rv_in, rv_out, S, 0, nb + rb, st));
  fill_rs_rec<<<kg_div_up(S, kThreads), kThreads, 0, st>>>(triplets, rv_out, S, reinterpret_cast<int4*>(rs_rec));
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" size_t kg_triplet_index_workspace_bytes(int n_triplets) {
  int S = n_triplets > 0 ? n_triplets : 1;
  return 2 * kg_align_up(((size_t)2 * S + 1) * 8) + 2 * kg_align_up(((size_t)2 * S + 1) * 4) +
         2 * kg_align_up(((size_t)S + 1) * 8) + 2 * kg_align_up(((size_t)S + 1) * 4) + triplet_cub_bytes(S) +
         kg_align_up(sizeof(unsigned) << orient_bits(S)) + 1024;
}

static int triplet_index_impl(const int32_t* triplets, int n_triplets, int n_nodes, int n_rels,
                              void* rs_rec, int32_t* ent_ptr, void* ent_pack, int ent_mode_req, void* workspace,
                              size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_triplets >= 0 && n_nodes > 0 && n_rels > 0, "triplet index: bad sizes");
  KG_REQUIRE(n_nodes < (1 << 24) && n_rels < (1 << 16), "triplet index: n_nodes < 2^24, n_rels < 2^16");
  cudaStream_t st = kg_stream(stream);
  const int S = n_triplets;
  if (S == 0) {
    if (ent_ptr) KG_CUDA(cudaMemsetAsync(ent_ptr, 0, sizeof(int) * (n_nodes + 1), st));
    return KG_OK;
  }
  KgArena ws(workspace, workspace_bytes);
  const int ent_mode = (ent_ptr != nullptr && ent_pack != nullptr) ? ent_mode_req : 0;   // the (entity, r) index is optional
  unsigned long long* ek_in = ws.take<unsigned long long>(2 * (size_t)S + 1);
  unsigned long long* ek_out = ws.take<unsigned long long>(2 * (size_t)S + 1);
  int* ev_in = ws.take<int>(2 * (size_t)S + 1);
  int* ev_out = ws.take<int>(2 * (size_t)S + 1);
  unsigned long long* rk_in = ws.take<unsigned long long>((size_t)S + 1);
  unsigned long long* rk_out = ws.take<unsigned long long>((size_t)S + 1);
  int* rv_in = ws.take<int>((size_t)S + 1);
  int* rv_out = ws.take<int>((size_t)S + 1);
  size_t temp_bytes = triplet_cub_bytes(S);
  void* temp = ws.take<char>(temp_bytes);
  const int obits = orient_bits(S);
  unsigned* table = ws.take<unsigned>((size_t)1 << obits);
  if (!ek_in || !ek_out || !ev_in || !ev_out || !rk_in || !rk_out || !rv_in || !rv_out || !temp || !table)
    return kg_fail(KG_ERR_WORKSPACE, "triplet index: workspace too small");
  const int nb = bits_for(n_nodes), rb = bits_for(n_rels);
  const bool orient = S >= (1 << 14);          // small batches: not worth the extra pass
  if (orient) {
    KG_CUDA(cudaMemsetAsync(table, 0, sizeof(unsigned) << obits, st));
    orient_count<<<kg_div_up(S, kThreads), kThreads, 0, st>>>(triplets, S, table, (1u << obits) - 1u);
    KG_LAUNCH_OK();
  }
  if (nb + rb <= 32)           // the 64-bit key buffers hold the 32-bit keys
    return triplet_sorts<unsigned>(triplets, S, n_nodes, nb, rb, orient ? table : nullptr, (1u << obits) - 1u, ent_mode,
                                   reinterpret_cast<unsigned*>(rk_in), reinterpret_cast<unsigned*>(rk_out), rv_in, rv_out,
                                   reinterpret_cast<unsigned*>(ek_in), reinterpret_cast<unsigned*>(ek_out), ev_in, ev_out,
                                   temp, temp_bytes, rs_rec, ent_ptr, ent_pack, st);
  return triplet_sorts<unsigned long long>(triplets, S, n_nodes, nb, rb, orient ? table : nullptr, (1u << obits) - 1u, ent_mode, rk_in, rk_out,
                                           rv_in, rv_out, ek_in, ek_out, ev_in, ev_out, temp, temp_bytes, rs_rec, ent_ptr,
                                           ent_pack, st);
}

extern "C" int kg_triplet_index(const int32_t* triplets, int n_triplets, int n_nodes, int n_rels,
                                void* rs_rec, int32_t* ent_ptr, void* ent_pack, void* workspace,
                                size_t workspace_bytes, void* stream) {
  return triplet_index_impl(triplets, n_triplets, n_nodes, n_rels, rs_rec, ent_ptr, ent_pack, 1, workspace, workspace_bytes,
                            stream);
}

// rs_rec as above plus the (trailing entity, r)-ordered index of the S triplets: trail_ptr [n_nodes + 1],
// trail_pack [S] int4 {leading entity, r, t, 0} - what kg_distmult_bwd_dz_trailing walks
extern "C" int kg_triplet_index_trailing(const int32_t* triplets, int n_triplets, int n_nodes, int n_rels,
                                         void* rs_rec, int32_t* trail_ptr, void* trail_pack, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  KG_REQUIRE(trail_ptr && trail_pack, "triplet index (trailing): null output");
  return triplet_index_impl(triplets, n_triplets, n_nodes, n_rels, rs_rec, trail_ptr, trail_pack, 2, workspace,
                            workspace_bytes, stream);
}

// ------------------------------------------------------------------------------------------
// (r, s)-ordered pass over the triplets, one warp per chunk of kChunkT consecutive records.
//   FUSED : score_t = sum_d (z[s,d] w[r,d]) z[o,d] + shift; BCE-with-logits term; g_t = (sigmoid - y) / S;
//           dw[r,:] += g_t z[s,:] z[o,:]          (link_predict.py:57-63,74-77 and their backward into w)
//   !FUSED: g_t given; dw only
// A lane keeps its float4 slots of w[r] and z[s] in registers while the run lasts, streams z[o]
// (2 KB, coalesced), and flushes the dw accumulators with vector reductions when r changes.
// ------------------------------------------------------------------------------------------
static constexpr int kChunkT = 32;

__device__ __forceinline__ void red_add_v4(float* addr, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

// DZ: 0 = no gradient wrt z; 1 = both ends (dz[o] reduced per triplet); 2 = leading end only (dz[s] over the run):
// the trailing end's gradient is then gathered by kg_distmult_bwd_dz_trailing - the form for a z that does not fit L2,
// where a reduction into a random row is a DRAM read-modify-write (4 KB of traffic) and a gather is a 2 KB read
template <int NV, bool FUSED, int DZ>
__global__ void __launch_bounds__(kThreads)
distmult_rs_kernel(const float* __restrict__ z, const float* __restrict__ w, const int4* __restrict__ rec,
                   const float* __restrict__ labels, const float* __restrict__ g_in,
                   const float* __restrict__ shift_p, int S, int h, float inv_S, float* __restrict__ score_out,
                   float* __restrict__ g_out, float* __restrict__ dw, float* __restrict__ dz,
                   float* __restrict__ loss_part, float* __restrict__ gsum_part) {
  const int warp = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  const int k0 = warp * kChunkT;
  if (k0 >= S) return;
  const int k1 = min(S, k0 + kChunkT), nvec = h >> 2;
  const float shift = (FUSED && shift_p) ? __ldg(shift_p) : 0.f;
  float4 zs[NV], wr[NV], acc[NV], acs[DZ ? NV : 1];   // acc: dw[r] of the run, acs: dz[s] of the run
#pragma unroll
  for (int i = 0; i < NV; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int i = 0; i < (DZ ? NV : 1); ++i) acs[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  int cs = -1, cr = -1;
  float loss = 0.f, gsum = 0.f;
  auto flush_s = [&]() {                      // dz[cs] += sum over the (r, s) run of g w[r] z[o]
    if (DZ && cs >= 0) {
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        if (c < nvec) red_add_v4(dz + (size_t)cs * h + 4 * c, acs[i]);
        acs[DZ ? i : 0] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
  };
  int4 rc = __ldg(rec + k0);
  for (int k = k0; k < k1; ++k) {
    const int4 nxt = k + 1 < k1 ? __ldg(rec + k + 1) : rc;      // prefetch the next record
    if (rc.y != cr) {
      flush_s();
      if (cr >= 0) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = lane + 32 * i;
          if (c < nvec) red_add_v4(dw + (size_t)cr * h + 4 * c, acc[i]);
          acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      cr = rc.y;
      cs = -1;
      if (FUSED || DZ) {
#pragma unroll
        for (int i = 0; i < NV; ++i) {
          const int c = lane + 32 * i;
          wr[i] = c < nvec ? __ldg(reinterpret_cast<const float4*>(w + (size_t)cr * h) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
    if (rc.x != cs) {
      flush_s();
      cs = rc.x;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        zs[i] = c < nvec ? __ldg(reinterpret_cast<const float4*>(z + (size_t)cs * h) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    float4 zo[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      zo[i] = c < nvec ? __ldg(reinterpret_cast<const float4*>(z + (size_t)rc.z * h) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float g;
    if (FUSED) {
      float dot = 0.f;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        dot = fmaf(zs[i].x * wr[i].x, zo[i].x, dot);
        dot = fmaf(zs[i].y * wr[i].y, zo[i].y, dot);
        dot = fmaf(zs[i].z * wr[i].z, zo[i].z, dot);
        dot = fmaf(zs[i].w * wr[i].w, zo[i].w, dot);
      }
      dot = kg_warp_sum(dot);
      const float xv = dot + shift, y = __ldg(labels + rc.w);
      // F.binary_cross_entropy_with_logits and its derivative from ONE fast exponential: t = e^{-|x|},
      // softplus(-|x|) = log(1 + t), sigmoid(x) = x >= 0 ? 1 / (1 + t) : t / (1 + t).  (Every lane computes
      // this per triplet, so it is kept to ~10 instructions; errors ~1e-7, far inside the 1e-4 bar.)
      const float t = __expf(-fabsf(xv)), inv1t = __frcp_rn(1.f + t);
      loss += fmaxf(xv, 0.f) - xv * y + __logf(1.f + t);
      g = ((xv >= 0.f ? inv1t : t * inv1t) - y) * inv_S;
      gsum += g;
      if (lane == 0) {
        g_out[rc.w] = g;
        if (score_out) score_out[rc.w] = xv;
      }
    } else {
      g = __ldg(g_in + rc.w);
    }
    if (DZ == 1) {                            // dz[o] += g w[r] z[s]: one coalesced 2 KB vector reduction per triplet
#pragma unroll
      for (int i = 0; i < NV; ++i) {
        const int c = lane + 32 * i;
        if (c < nvec)
          red_add_v4(dz + (size_t)rc.z * h + 4 * c,
                     make_float4(g * wr[i].x * zs[i].x, g * wr[i].y * zs[i].y, g * wr[i].z * zs[i].z, g * wr[i].w * zs[i].w));
      }
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float tx = g * zo[i].x, ty = g * zo[i].y, tz = g * zo[i].z, tw = g * zo[i].w;
      acc[i].x = fmaf(tx, zs[i].x, acc[i].x);
      acc[i].y = fmaf(ty, zs[i].y, acc[i].y);
      acc[i].z = fmaf(tz, zs[i].z, acc[i].z);
      acc[i].w = fmaf(tw, zs[i].w, acc[i].w);
      if (DZ) {
        acs[DZ ? i : 0].x = fmaf(tx, wr[i].x, acs[DZ ? i : 0].x);
        acs[DZ ? i : 0].y = fmaf(ty, wr[i].y, acs[DZ ? i : 0].y);
        acs[DZ ? i : 0].z = fmaf(tz, wr[i].z, acs[DZ ? i : 0].z);
        acs[DZ ? i : 0].w = fmaf(tw, wr[i].w, acs[DZ ? i : 0].w);
      }
    }
    rc = nxt;
  }
  flush_s();
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < nvec) red_add_v4(dw + (size_t)cr * h + 4 * c, acc[i]);
  }
  if (FUSED && lane == 0) {
    loss_part[warp] = loss;
    gsum_part[warp] = gsum;
  }
}

// scalar variant for h % 4 != 0 or unaligned rows (no register caching)
template <bool FUSED>
__global__ void __launch_bounds__(kThreads)
distmult_rs_generic(const float* __restrict__ z, const float* __restrict__ w, const int4* __restrict__ rec,
                    const float* __restrict__ labels, const float* __restrict__ g_in,
                    const float* __restrict__ shift_p, int S, int h, float inv_S, float* __restrict__ score_out,
                    float* __restrict__ g_out, float* __restrict__ dw, float* __restrict__ dz,
                    float* __restrict__ loss_part, float* __restrict__ gsum_part) {
  const int warp = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  const int k0 = warp * kChunkT;
  if (k0 >= S) return;
  const int k1 = min(S, k0 + kChunkT);
  const float shift = (FUSED && shift_p) ? __ldg(shift_p) : 0.f;
  float loss = 0.f, gsum = 0.f;
  for (int k = k0; k < k1; ++k) {
    const int4 rc = __ldg(rec + k);
    const float* zs = z + (size_t)rc.x * h;
    const float* wr = w + (size_t)rc.y * h;
    const float* zo = z + (size_t)rc.z * h;
    float g;
    if (FUSED) {
      float dot = 0.f;
      for (int c = lane; c < h; c += 32) dot = fmaf(__ldg(zs + c) * __ldg(wr + c), __ldg(zo + c), dot);
      dot = kg_warp_sum(dot);
      const float xv = dot + shift, y = __ldg(labels + rc.w);
      loss += fmaxf(xv, 0.f) - xv * y + log1pf(expf(-fabsf(xv)));
      g = (kg_sigmoid(xv) - y) * inv_S;
      gsum += g;
      if (lane == 0) {
        g_out[rc.w] = g;
        if (score_out) score_out[rc.w] = xv;
      }
    } else {
      g = __ldg(g_in + rc.w);
    }
    for (int c = lane; c < h; c += 32) {
      const float a = __ldg(zs + c), b = __ldg(zo + c);
      atomicAdd(dw + (size_t)rc.y * h + c, g * a * b);
      if (dz) {
        const float wv = __ldg(w + (size_t)rc.y * h + c);
        atomicAdd(dz + (size_t)rc.x * h + c, g * wv * b);
        atomicAdd(dz + (size_t)rc.z * h + c, g * wv * a);
      }
    }
  }
  if (FUSED && lane == 0) {
    loss_part[warp] = loss;
    gsum_part[warp] = gsum;
  }
}

template <bool FUSED>
static int launch_rs(const float* z, const float* w, const void* rs_rec, const float* labels, const float* g_in,
                     const float* shift, int S, int h, float* score_out, float* g_out, float* dw, float* dz,
                     float* loss_part, float* gsum_part, cudaStream_t st, bool lead_only = false) {
  const int warps = kg_div_up(S, kChunkT);
  const int grid = kg_div_up((long long)warps * 32, kThreads);
  const int4* rec = reinterpret_cast<const int4*>(rs_rec);
  const float inv_S = 1.0f / (float)S;
  const bool vec = (h % 4 == 0) && h <= 1024 &&
                   ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(dw) |
                     reinterpret_cast<uintptr_t>(dz)) & 15) == 0;
#define KG_RS_LAUNCH(NV_)                                                                                       \
  do {                                                                                                          \
    if (dz && lead_only)                                                                                        \
      distmult_rs_kernel<NV_, FUSED, 2><<<grid, kThreads, 0, st>>>(z, w, rec, labels, g_in, shift, S, h, inv_S,    \
                                                                   score_out, g_out, dw, dz, loss_part, gsum_part); \
    else if (dz)                                                                                                \
      distmult_rs_kernel<NV_, FUSED, 1><<<grid, kThreads, 0, st>>>(z, w, rec, labels, g_in, shift, S, h, inv_S,    \
                                                                   score_out, g_out, dw, dz, loss_part, gsum_part); \
    else                                                                                                        \
      distmult_rs_kernel<NV_, FUSED, 0><<<grid, kThreads, 0, st>>>(z, w, rec, labels, g_in, shift, S, h, inv_S,    \
                                                                   score_out, g_out, dw, dz, loss_part, gsum_part); \
  } while (0)
  if (!vec) distmult_rs_generic<FUSED><<<grid, kThreads, 0, st>>>(z, w, rec, labels, g_in, shift, S, h, inv_S, score_out, g_out, dw, dz, loss_part, gsum_part);
  else if (h <= 128) KG_RS_LAUNCH(1);
  else if (h <= 256) KG_RS_LAUNCH(2);
  else if (h <= 512) KG_RS_LAUNCH(4);
  else KG_RS_LAUNCH(8);
#undef KG_RS_LAUNCH
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" size_t kg_distmult_bce_workspace_bytes(int n_triplets) {
  const size_t warps = (size_t)kg_div_up(n_triplets > 0 ? n_triplets : 1, kChunkT);
  return 2 * kg_align_up(warps * sizeof(float)) + kg_align_up(sizeof(float) * kMaxPartials) + 1024;
}

// Fused DistMult score + BCE-with-logits (mean) + gradient wrt the score and wrt w_relation.
//   loss_out[0] = mean_t BCE(score_t, labels_t);  gsum_out[0] = sum_t g_t (gradient wrt the scalar shift)
//   g_out[t] = dloss/dscore_t;  dw (zero-filled by the caller) += sum_t g_t z[s_t] z[o_t];  score_out optional
//   dz (optional, zero-filled by the caller) += sum_t g_t w[r_t] (z[o_t] into row s_t, z[s_t] into row o_t):
//   the whole backward into z in the same pass - z[o] is in registers anyway, dz[s] is kept in registers over
//   an (r, s) run and dz[o] goes out as one coalesced 2 KB vector reduction per triplet
static int distmult_bce_impl(const float* z, const float* w, const void* rs_rec, const float* labels,
                             int n_triplets, int h, const float* shift, float* score_out, float* g_out,
                             float* dw, float* dz, float* loss_out, float* gsum_out, void* workspace,
                             size_t workspace_bytes, void* stream, bool lead_only) {
  KG_REQUIRE(n_triplets >= 0 && h > 0, "distmult bce: bad sizes");
  if (lead_only)
    KG_REQUIRE(dz && h % 4 == 0 && h <= 1024 &&
                   ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(dw) |
                     reinterpret_cast<uintptr_t>(dz)) & 15) == 0,
               "distmult bce (leading end): needs dz, h % 4 == 0, h <= 1024 and 16-byte aligned rows");
  cudaStream_t st = kg_stream(stream);
  if (n_triplets == 0) {
    KG_CUDA(cudaMemsetAsync(loss_out, 0, sizeof(float), st));
    KG_CUDA(cudaMemsetAsync(gsum_out, 0, sizeof(float), st));
    return KG_OK;
  }
  const size_t warps = (size_t)kg_div_up(n_triplets, kChunkT);
  KgArena ws(workspace, workspace_bytes);
  float* loss_part = ws.take<float>(warps);
  float* gsum_part = ws.take<float>(warps);
  float* red = ws.take<float>(kMaxPartials);
  if (!loss_part || !gsum_part || !red) return kg_fail(KG_ERR_WORKSPACE, "distmult bce: workspace too small");
  int rc = launch_rs<true>(z, w, rs_rec, labels, nullptr, shift, n_triplets, h, score_out, g_out, dw, dz, loss_part,
                           gsum_part, st, lead_only);
  if (rc != KG_OK) return rc;
  rc = run_reduce(loss_part, nullptr, (long long)warps, 0, 1.0f / (float)n_triplets, 0.f, nullptr, loss_out, red,
                  sizeof(float) * kMaxPartials, st);
  if (rc != KG_OK) return rc;
  return run_reduce(gsum_part, nullptr, (long long)warps, 0, 1.f, 0.f, nullptr, gsum_out, red,
                    sizeof(float) * kMaxPartials, st);
}

extern "C" int kg_distmult_bce_fwd(const float* z, const float* w, const void* rs_rec, const float* labels,
                                   int n_triplets, int h, const float* shift, float* score_out, float* g_out,
                                   float* dw, float* dz, float* loss_out, float* gsum_out, void* workspace,
                                   size_t workspace_bytes, void* stream) {
  return distmult_bce_impl(z, w, rs_rec, labels, n_triplets, h, shift, score_out, g_out, dw, dz, loss_out, gsum_out,
                           workspace, workspace_bytes, stream, false);
}

// The same pass with only the LEADING end's share of dz (the entity each rs_rec run keeps in registers):
//   dz[lead_t] += g_t w[r_t] z[trail_t];   the trailing end's share is kg_distmult_bwd_dz_trailing's.
// For a z that does not fit L2: a reduction into a random row is then a DRAM read-modify-write.
extern "C" int kg_distmult_bce_fwd_lead(const float* z, const float* w, const void* rs_rec, const float* labels,
                                        int n_triplets, int h, const float* shift, float* score_out, float* g_out,
                                        float* dw, float* dz, float* loss_out, float* gsum_out, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  return distmult_bce_impl(z, w, rs_rec, labels, n_triplets, h, shift, score_out, g_out, dw, dz, loss_out, gsum_out,
                           workspace, workspace_bytes, stream, true);
}

// dw[r,:] += sum_{t: rel_t = r} gscore[t] * z[s_t,:] * z[o_t,:]; dw zero-filled by the caller
extern "C" int kg_distmult_bwd_dw(const float* z, const float* gscore, const void* rs_rec, int n_triplets, int h,
                                  float* dw, void* stream) {
  KG_REQUIRE(n_triplets >= 0 && h > 0, "distmult dw: bad sizes");
  if (n_triplets == 0) return KG_OK;
  return launch_rs<false>(z, nullptr, rs_rec, nullptr, gscore, nullptr, n_triplets, h, nullptr, nullptr, dw, nullptr,
                          nullptr, nullptr, kg_stream(stream));
}

// ------------------------------------------------------------------------------------------
// dz[v, :] = sum over the (entity, r)-ordered index of gscore[t] * w[r, :] * z[other, :]
// one thread per (entity, VEC consecutive columns); w[r] stays in registers while r repeats; no atomics
// ------------------------------------------------------------------------------------------
template <int VEC, bool ACC>
__global__ void __launch_bounds__(kThreads)
distmult_dz_kernel(const float* __restrict__ z, const float* __restrict__ w,
                   const float* __restrict__ gscore, const int* __restrict__ ent_ptr,
                   const int4* __restrict__ ent_pack, int n_nodes, int h, float* __restrict__ dz) {
  const int cols = h / VEC;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n_nodes * cols) return;
  const int v = (int)(t / cols), c = (int)(t % cols);
  const int e_end = __ldg(ent_ptr + v + 1);
  float acc[VEC];
#pragma unroll
  for (int q = 0; q < VEC; ++q) acc[q] = 0.f;
  int cr = -1;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 2
  for (int e = __ldg(ent_ptr + v); e < e_end; ++e) {
    const int4 p = __ldg(ent_pack + e);          // {other, rel, triplet, -}
    const float g = __ldg(gscore + p.z);
    if (p.y != cr) {
      cr = p.y;
      if (VEC == 4) a = __ldg(reinterpret_cast<const float4*>(w + (size_t)cr * h) + c);
      else a.x = __ldg(w + (size_t)cr * h + c);
    }
    if (VEC == 4) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(z + (size_t)p.x * h) + c);
      acc[0] = fmaf(g * a.x, b.x, acc[0]);
      acc[1 % VEC] = fmaf(g * a.y, b.y, acc[1 % VEC]);
      acc[2 % VEC] = fmaf(g * a.z, b.z, acc[2 % VEC]);
      acc[3 % VEC] = fmaf(g * a.w, b.w, acc[3 % VEC]);
    } else {
      acc[0] = fmaf(g * a.x, __ldg(z + (size_t)p.x * h + c), acc[0]);
    }
  }
  if (ACC && e_end == __ldg(ent_ptr + v)) return;     // nothing to add to this row
  if (VEC == 4) {
    float4* p4 = reinterpret_cast<float4*>(dz + (size_t)v * h) + c;
    float4 o4 = make_float4(acc[0], acc[1 % VEC], acc[2 % VEC], acc[3 % VEC]);
    if (ACC) { const float4 q = *p4; o4.x += q.x; o4.y += q.y; o4.z += q.z; o4.w += q.w; }
    *p4 = o4;
  } else {
    dz[(size_t)v * h + c] = ACC ? dz[(size_t)v * h + c] + acc[0] : acc[0];
  }
}

template <bool ACC>
static int launch_dz(const float* z, const float* w, const float* gscore, const int32_t* ent_ptr, const void* ent_pack,
                     int n_nodes, int h, float* dz, void* stream) {
  KG_REQUIRE(n_nodes >= 0 && h > 0, "distmult dz: bad sizes");
  if (n_nodes == 0) return KG_OK;
  const bool vec = (h % 4 == 0) &&
                   ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(dz)) & 15) == 0;
  const int4* pk = reinterpret_cast<const int4*>(ent_pack);
  if (vec) {
    distmult_dz_kernel<4, ACC><<<kg_div_up((long long)n_nodes * (h / 4), kThreads), kThreads, 0, kg_stream(stream)>>>(
        z, w, gscore, ent_ptr, pk, n_nodes, h, dz);
  } else {
    distmult_dz_kernel<1, ACC><<<kg_div_up((long long)n_nodes * h, kThreads), kThreads, 0, kg_stream(stream)>>>(
        z, w, gscore, ent_ptr, pk, n_nodes, h, dz);
  }
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" int kg_distmult_bwd_dz(const float* z, const float* w, const float* gscore,
                                  const int32_t* ent_ptr, const void* ent_pack, int n_nodes, int h,
                                  float* dz, void* stream) {
  return launch_dz<false>(z, w, gscore, ent_ptr, ent_pack, n_nodes, h, dz, stream);
}

// dz[v, :] += sum over the triplets whose TRAILING end is v of gscore[t] * w[r, :] * z[leading end, :]
// (kg_triplet_index_trailing's index; each row has one owner thread group: plain loads and stores, no atomics,
// a fixed summation order).  Completes kg_distmult_bce_fwd_lead.
extern "C" int kg_distmult_bwd_dz_trailing(const float* z, const float* w, const float* gscore,
                                           const int32_t* trail_ptr, const void* trail_pack, int n_nodes, int h,
                                           float* dz, void* stream) {
  return launch_dz<true>(z, w, gscore, trail_ptr, trail_pack, n_nodes, h, dz, stream);
}
