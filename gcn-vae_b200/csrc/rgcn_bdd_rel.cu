// a3: RelGraphConv(regularizer="bdd") message passing over relation-sorted edge records
// {src, dst, etype, norm} (kg_graph_index / kg_graph_rel_tiled), C entry points.  A call runs the
// first kernel family that takes its block shape:
//   1. block-owner kernels (rgcn_bdd_warp.cuh): 5x5 blocks (B % 4 == 0, B <= 128) and 5x10 blocks
//      (B even, B <= 128), straight from the DGL-layout weight.  The only family for peer row
//      blocks and for column chunks (the _cols entry points).
//   2. register-tile kernels (rgcn_bdd_tile.cuh): blocks whose sides divide by 4, 5, 8, 10, 20, 25
//      or 50, on the derived w_fwd / w_bwd layouts (kg_bdd_weight_layouts).  Backward is two
//      launches: dX (the forward kernel on the transposed layout), then dW.
//   3. the generic pair below: any shape whose relation weights fit in shared memory.
#include "common.cuh"

#include "rgcn_bdd_own.cuh"
#include "rgcn_bdd_tile.cuh"
#include "rgcn_bdd_warp.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kChunk = 128;   // consecutive relation-sorted edges per CTA

// hints (bit mask) of the C entry points: which gathered matrix is streamed from HBM (larger than
// L2, every row used about once) and should not displace the L2-resident reduction tile
constexpr int kHintStreamD = 2;

// ------------------------------------------------------------------------------------------
// any block shape: run-time FI/FO, scalar reductions, dW accumulated in shared memory
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void stage_row_any(float* dst, const float* __restrict__ src, int n) {
  for (int i = threadIdx.x; i < n; i += kThreads) dst[i] = __ldg(src + i);
}

__global__ void __launch_bounds__(kThreads)
bdd_rel_scatter_generic(const float* __restrict__ feat, const int4* __restrict__ pack, int E,
                        const float* __restrict__ wl, int B, int FI, int FO, int swap, float* __restrict__ out) {
  extern __shared__ __align__(16) float sm[];
  const int width = B * FO, in_w = B * FI;
  float* W_s = sm;
  float* X_s = sm + FI * width;
  const int e0 = blockIdx.x * kChunk, e1 = min(E, e0 + kChunk);
  int cur = -1;
  for (int e = e0; e < e1; ++e) {
    const int4 p = __ldg(pack + e);
    __syncthreads();
    if (p.z != cur) {
      stage_row_any(W_s, wl + (size_t)p.z * FI * width, FI * width);
      cur = p.z;
    }
    stage_row_any(X_s, feat + (size_t)(swap ? p.y : p.x) * in_w, in_w);
    __syncthreads();
    const float nv = __int_as_float(p.w);
    float* orow = out + (size_t)(swap ? p.x : p.y) * width;
    for (int j = threadIdx.x; j < width; j += kThreads) {
      const float* xs = X_s + (j / FO) * FI;
      float m = 0.f;
      for (int i = 0; i < FI; ++i) m = fmaf(xs[i], W_s[i * width + j], m);
      atomicAdd(orow + j, nv * m);
    }
  }
}

__global__ void __launch_bounds__(kThreads)
bdd_rel_backward_generic(const float* __restrict__ x, const float* __restrict__ dagg,
                         const int4* __restrict__ pack, int E, const float* __restrict__ w_bwd, int B, int SI,
                         int SO, float* __restrict__ dx, float* __restrict__ dW) {
  extern __shared__ __align__(16) float sm[];
  const int in_w = B * SI, out_w = B * SO, KW = B * SI * SO;
  float* W_s = sm;                 // [SO][in_w]
  float* A_s = W_s + SO * in_w;    // [KW] weight-gradient accumulators of the current relation
  float* X_s = A_s + KW;           // [in_w]
  float* D_s = X_s + in_w;         // [out_w]
  const int e0 = blockIdx.x * kChunk, e1 = min(E, e0 + kChunk);
  int cur = -1;
  for (int e = e0; e < e1; ++e) {
    const int4 p = __ldg(pack + e);
    __syncthreads();
    if (p.z != cur) {
      for (int k = threadIdx.x; k < KW; k += kThreads) {
        if (cur >= 0) atomicAdd(dW + (size_t)cur * KW + k, A_s[k]);
        A_s[k] = 0.f;
      }
      stage_row_any(W_s, w_bwd + (size_t)p.z * SO * in_w, SO * in_w);
      cur = p.z;
    }
    stage_row_any(X_s, x + (size_t)p.x * in_w, in_w);
    stage_row_any(D_s, dagg + (size_t)p.y * out_w, out_w);
    __syncthreads();
    const float nv = __int_as_float(p.w);
    for (int k = threadIdx.x; k < KW; k += kThreads) {
      const int b = k / (SI * SO), rem = k - b * (SI * SO);
      A_s[k] = fmaf(nv * X_s[b * SI + rem / SO], D_s[b * SO + rem % SO], A_s[k]);
    }
    if (dx) {
      float* drow = dx + (size_t)p.x * in_w;
      for (int j = threadIdx.x; j < in_w; j += kThreads) {
        const float* ds = D_s + (j / SI) * SO;
        float m = 0.f;
        for (int o = 0; o < SO; ++o) m = fmaf(ds[o], W_s[o * in_w + j], m);
        atomicAdd(drow + j, nv * m);
      }
    }
  }
  __syncthreads();
  if (cur >= 0)
    for (int k = threadIdx.x; k < KW; k += kThreads) atomicAdd(dW + (size_t)cur * KW + k, A_s[k]);
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace

// 1 when kg_bdd_rel_fwd / kg_bdd_rel_bwd need the derived layouts of kg_bdd_weight_layouts for this
// shape, 0 when they read the DGL-layout weight directly (block-owner kernels, rgcn_bdd_own.cuh)
extern "C" int kg_bdd_layouts_needed(int num_bases, int si, int so) {
  return bddown::eligible(num_bases, si, so) ? 0 : 1;
}

// agg[dst] += norm * blockdiag(W[etype]) x[src] over relation-sorted edges; agg zero-filled by the caller
extern "C" int kg_bdd_rel_fwd(const float* x, const void* x_parts, int part_rows, const void* rel_pack,
                              int n_edges, const float* weight, const float* w_fwd, int num_bases, int si,
                              int so, float* agg, int hints, void* stream) {
  KG_REQUIRE(n_edges >= 0 && num_bases > 0 && si > 0 && so > 0, "bdd rel fwd: bad sizes");
  KG_REQUIRE(x_parts == nullptr || part_rows > 0, "bdd rel fwd: part_rows must be positive");
  if (n_edges == 0) return KG_OK;
  cudaStream_t st = kg_stream(stream);
  if (weight && bddown::eligible(num_bases, si, so) && aligned16(x) && aligned16(weight) && aligned16(agg)) {
    const bddown::RowSource src{x, reinterpret_cast<const float* const*>(x_parts), part_rows};
    // (gather ring depth, reductions in flight per warp) = (4, 2) / (8, 2): a sweep at the wikikg2 shape
    // (profiles/r02g_reduction_depth_sweep.txt) found 3-6 reductions in flight no faster - the 5x10 launch sits at
    // 84 % of what L2 sustains for whole-row reductions (kg_probe_l2), not on the latency of a bulk reduction
    if (so == 5) return bddwarp::launch_fwd<5, 5, 4, 1, 4>(src, rel_pack, n_edges, weight, num_bases, hints, agg, st);
    return bddwarp::launch_fwd<5, 10, 2, 2, 8>(src, rel_pack, n_edges, weight, num_bases, hints, agg, st);
  }
  KG_REQUIRE(x_parts == nullptr, "bdd rel fwd: peer row blocks need the 5x5 / 5x10 block-owner kernels");
  KG_REQUIRE(w_fwd != nullptr, "bdd rel fwd: this block shape needs the w_fwd layout (kg_bdd_weight_layouts)");
  if (bddtile::eligible(num_bases, si, so) && aligned16(x) && aligned16(w_fwd) && aligned16(agg))
    return bddtile::launch_fwd(x, rel_pack, n_edges, w_fwd, si, so, num_bases, 0, agg, st);
  const size_t smem = sizeof(float) * ((size_t)si * num_bases * so + (size_t)num_bases * si);
  KG_REQUIRE(smem <= 200 * 1024, "bdd rel fwd: block weights of one relation exceed shared memory");
  KG_CUDA(cudaFuncSetAttribute(bdd_rel_scatter_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bdd_rel_scatter_generic<<<kg_div_up(n_edges, kChunk), kThreads, smem, st>>>(
      x, reinterpret_cast<const int4*>(rel_pack), n_edges, w_fwd, num_bases, si, so, 0, agg);
  KG_LAUNCH_OK();
  return KG_OK;
}

// dx (zero-filled, may be NULL) and dweight (zero-filled) of the same layer
extern "C" int kg_bdd_rel_bwd(const float* x, const void* x_parts, int part_rows, const float* dagg,
                              const void* rel_pack, int n_edges, const float* weight, const float* w_bwd,
                              int num_bases, int si, int so, float* dx, float* dweight, int hints,
                              void* stream) {
  KG_REQUIRE(n_edges >= 0 && num_bases > 0 && si > 0 && so > 0, "bdd rel bwd: bad sizes");
  KG_REQUIRE(x_parts == nullptr || part_rows > 0, "bdd rel bwd: part_rows must be positive");
  if (n_edges == 0) return KG_OK;
  cudaStream_t st = kg_stream(stream);
  if (weight && bddown::eligible(num_bases, si, so) && aligned16(x) && aligned16(dagg) && aligned16(weight) &&
      aligned16(dx) && aligned16(dweight)) {
    const bddown::RowSource src{x, reinterpret_cast<const float* const*>(x_parts), part_rows};
    // dagg streams from HBM (wikikg2 shape): with 5x5 blocks the partner warps of the paired variant share one
    // gather of dagg[dst] (103 GB of DRAM traffic instead of 148 GB, 25.0 vs 25.3 ms); with 5x10 blocks the two
    // variants time the same in the bench loop (48.7 vs 49.6 ms; under ncu 40.1 vs 46.1 ms), so the independent
    // warps - no cross-warp handshake - serve every regime
    if ((hints & kHintStreamD) && so == 5)
      return bddwarp::launch_bwd_paired<5, 5, 4, 1, 6>(src, dagg, rel_pack, n_edges, weight, num_bases, hints, dx, dweight, st);
    if (so == 5)
      return bddwarp::launch_bwd<5, 5, 4, 1, 4>(src, dagg, rel_pack, n_edges, weight, num_bases, hints, dx, dweight, st);
    return bddwarp::launch_bwd<5, 10, 2, 2, 4>(src, dagg, rel_pack, n_edges, weight, num_bases, hints, dx, dweight, st);
  }
  KG_REQUIRE(x_parts == nullptr, "bdd rel bwd: peer row blocks need the 5x5 / 5x10 block-owner kernels");
  KG_REQUIRE(w_bwd != nullptr, "bdd rel bwd: this block shape needs the w_bwd layout (kg_bdd_weight_layouts)");
  if (bddtile::eligible(num_bases, si, so) && aligned16(x) && aligned16(dagg) && aligned16(w_bwd) &&
      aligned16(dx) && aligned16(dweight)) {
    if (dx != nullptr) {
      const int rc = bddtile::launch_fwd(dagg, rel_pack, n_edges, w_bwd, so, si, num_bases, 1, dx, st);
      if (rc != KG_OK) return rc;
    }
    return bddtile::launch_dw(x, dagg, rel_pack, n_edges, si, so, num_bases, dweight, st);
  }
  const int in_w = num_bases * si, out_w = num_bases * so;
  const size_t smem = sizeof(float) * ((size_t)so * in_w + (size_t)num_bases * si * so + in_w + out_w);
  KG_REQUIRE(smem <= 200 * 1024, "bdd rel bwd: block weights of one relation exceed shared memory");
  KG_CUDA(cudaFuncSetAttribute(bdd_rel_backward_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bdd_rel_backward_generic<<<kg_div_up(n_edges, kChunk), kThreads, smem, st>>>(
      x, dagg, reinterpret_cast<const int4*>(rel_pack), n_edges, w_bwd, num_bases, si, so, dx, dweight);
  KG_LAUNCH_OK();
  return KG_OK;
}


// ------------------------------------------------------------------------------------------
// Column chunks of a layer (destination-partitioned training pipelines message passing against
// column chunks of the layer-input all-gather and of the source-gradient reduce-scatter).
// The weight of a relation is block-diagonal, so blocks [block0, block0 + num_bases) of
// num_bases_total only touch columns [block0 * si, ...) of x and [block0 * so, ...) of agg:
//   x_chunk   [n_src, num_bases * si]   compact matrix holding just those columns (all nodes)
//   weight    the FULL weight [R, num_bases_total * si * so];  agg / dagg the FULL matrices
//   dx_chunk  [n_src, num_bases * si]   compact, zero-filled;  dweight the FULL gradient (zero-filled once)
// 5x5 / 5x10 blocks only (the warp-autonomous kernels).  A chunk is run with TWO blocks per lane and ONE warp per
// edge (the full layer uses 4 blocks per lane for 5x5 and two warps per edge for 5x10): num_bases even, <= 64, so
// that a chunk of about half the layer still fills 25 of a warp's 32 lanes.
// ------------------------------------------------------------------------------------------
extern "C" int kg_bdd_rel_fwd_cols(const float* x_chunk, const void* rel_pack, int n_edges, const float* weight,
                                   int block0, int num_bases, int num_bases_total, int si, int so, float* agg,
                                   int hints, void* stream) {
  KG_REQUIRE(n_edges >= 0 && num_bases > 0 && block0 >= 0 && block0 + num_bases <= num_bases_total, "bdd fwd cols: bad block range");
  KG_REQUIRE(si == 5 && (so == 5 || so == 10) && num_bases % 2 == 0 && num_bases <= 64 && aligned16(x_chunk) &&
             aligned16(weight) && aligned16(agg) && (block0 * si * so) % 4 == 0 && (block0 * so) % 4 == 0 &&
             (num_bases * si) % 4 == 0,
             "bdd fwd cols: needs 5x5 / 5x10 blocks, an even chunk of <= 64 blocks and 16-byte aligned chunk offsets");
  if (n_edges == 0) return KG_OK;
  cudaStream_t st = kg_stream(stream);
  const bddown::RowSource src{x_chunk, nullptr, 0};
  const float* w = weight + (size_t)block0 * si * so;
  float* out = agg + (size_t)block0 * so;
  const int ldw = num_bases_total * si * so, ldo = num_bases_total * so;
  if (so == 5) return bddwarp::launch_fwd<5, 5, 2, 1, 4>(src, rel_pack, n_edges, w, num_bases, hints, out, st, ldw, ldo);
  return bddwarp::launch_fwd<5, 10, 2, 1, 4>(src, rel_pack, n_edges, w, num_bases, hints, out, st, ldw, ldo);
}

extern "C" int kg_bdd_rel_bwd_cols(const float* x_chunk, const float* dagg, const void* rel_pack, int n_edges,
                                   const float* weight, int block0, int num_bases, int num_bases_total, int si,
                                   int so, float* dx_chunk, float* dweight, int hints, void* stream) {
  KG_REQUIRE(n_edges >= 0 && num_bases > 0 && block0 >= 0 && block0 + num_bases <= num_bases_total, "bdd bwd cols: bad block range");
  KG_REQUIRE(si == 5 && (so == 5 || so == 10) && num_bases % 2 == 0 && num_bases <= 64 && aligned16(x_chunk) &&
             aligned16(dagg) && aligned16(weight) && aligned16(dx_chunk) && aligned16(dweight) &&
             (block0 * si * so) % 4 == 0 && (block0 * so) % 4 == 0 && (num_bases * si) % 4 == 0,
             "bdd bwd cols: needs 5x5 / 5x10 blocks, an even chunk of <= 64 blocks and 16-byte aligned chunk offsets");
  if (n_edges == 0) return KG_OK;
  cudaStream_t st = kg_stream(stream);
  const bddown::RowSource src{x_chunk, nullptr, 0};
  const float* w = weight + (size_t)block0 * si * so;
  float* dw = dweight + (size_t)block0 * si * so;
  const float* dg = dagg + (size_t)block0 * so;
  const int ldw = num_bases_total * si * so, ldd = num_bases_total * so;
  if (so == 5)
    return bddwarp::launch_bwd<5, 5, 2, 1, 4>(src, dg, rel_pack, n_edges, w, num_bases, hints, dx_chunk, dw, st, ldw, ldd);
  return bddwarp::launch_bwd<5, 10, 2, 1, 4>(src, dg, rel_pack, n_edges, w, num_bases, hints, dx_chunk, dw, st, ldw, ldd);
}
