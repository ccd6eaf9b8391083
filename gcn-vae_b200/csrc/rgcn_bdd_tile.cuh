// a3: RelGraphConv(regularizer="bdd") message passing with register tiles, for diagonal blocks from
// 4x4 to 50x100 whose sides divide by 4, 5, 8, 10, 20, 25 or 50 (pick_tile): e.g. num_bases 10 .. 50
// at h = 500 (DGL RelGraphConv as constructed at kgvae/model.py:54-59 with a small --n-bases, such as
// the WN18 shape where DGL clamps num_bases to the 36 directed relation types).  The reference model's
// 5x5 and 5x10 blocks run on the block-owner kernels (rgcn_bdd_warp.cuh) while they fit there.
//
// Edges are walked in RELATION-MAJOR order.  Per edge the layer needs the whole block-diagonal weight
// of the edge's relation: B*si*so floats (10 KB for 5x5 blocks, 20 KB for 5x10) against a 2 KB source
// row.  Walking edges in destination order (rgcn_bdd.cu, first version) re-reads those weights from L2
// for every edge - 5-10x the feature bytes.  Here edges are walked in (node tile, relation) order - the
// etype-major record lists kg_graph_index / kg_graph_rel_tiled build - so that
//   * the threads of a slot keep the relation's weight in REGISTERS for a whole run of edges (no
//     per-edge weight traffic at all, not even shared memory), and
//   * the rows that are reduced into (out[dst] forward, dx[src] backward) belong to one node tile
//     sized to stay L2-resident, so the vector reductions never reach HBM and the only per-edge
//     HBM traffic is the gathered row (forward: x[src]; backward: dagg[dst]).
//
// A CTA takes 128 consecutive records (copied to shared memory once - no dependent index loads in
// the loop) and splits into independent SLOTS of whole warps, one edge per slot at a time; every
// slot runs its own 4-deep cp.async ring of gathered rows and synchronises with a named barrier, so
// there is no CTA-wide barrier in the loop.  Summation order across CTAs is not fixed: results are
// reproducible to fp32 rounding.
//
// The register tiling is two-dimensional so that a relation's WHOLE block-diagonal weight (B*si*so
// floats, up to 50 000) stays in the registers of the threads of one slot while the relation lasts:
//
//   forward / dX   a thread owns CO consecutive output columns (inside one block) and KI of the
//                  block's K input rows: w[KI][CO] registers, KI shared-memory broadcasts and
//                  KI*CO FMAs per edge, one vector reduction (red.v4 / red.v2 / red) of CO partial
//                  sums.  K-split threads (KS = K / KI > 1) reduce separately: the adds commute.
//   dW             a thread owns a TI x TO tile of one block's outer product x[src] (x) dagg[dst]
//                  in registers and flushes it with vector reductions when the relation changes.
//
// dX runs the forward kernel on the transposed layout (gathers dagg[dst], reduces into dx[src]).
#pragma once
#include "common.cuh"

namespace bddtile {

constexpr int kChunk = 128;   // consecutive relation-sorted edges per CTA
constexpr int kDepth = 4;     // gathered rows in flight per slot

__device__ __forceinline__ void cp16(float* dst, const float* __restrict__ src) {
  const uint32_t d = static_cast<uint32_t>(__cvta_generic_to_shared(dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(src) : "memory");
}
__device__ __forceinline__ void commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void slot_bar(int slot, int n) {
  asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "r"(n) : "memory");
}
template <int CO>
__device__ __forceinline__ void red_vec(float* addr, const float (&m)[CO], float s) {
  if constexpr (CO == 4)
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(s * m[0]), "f"(s * m[1]),
                 "f"(s * m[2]), "f"(s * m[3]) : "memory");
  else if constexpr (CO == 2)
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(s * m[0]), "f"(s * m[1]) : "memory");
  else
    atomicAdd(addr, s * m[0]);
}
// N consecutive floats from shared memory; `vec` = widest load (1, 2, 4 floats) the address allows
template <int N>
__device__ __forceinline__ void lds_n(float (&v)[N], const float* p, int vec) {
  if (N % 4 == 0 && vec == 4) {  // (N is a compile-time constant: dead branches fold away)
#pragma unroll
    for (int i = 0; i < N; i += 4) {
      const float4 t = *reinterpret_cast<const float4*>(p + i);
      v[i] = t.x; v[i + 1] = t.y; v[i + 2] = t.z; v[i + 3] = t.w;
    }
  } else if (N % 2 == 0 && vec >= 2) {
#pragma unroll
    for (int i = 0; i < N; i += 2) {
      const float2 t = *reinterpret_cast<const float2*>(p + i);
      v[i] = t.x; v[i + 1] = t.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < N; ++i) v[i] = p[i];
  }
}
__device__ __forceinline__ const float* row32(const float* base, int row, int width) {
  return base + (size_t)(unsigned)row * (unsigned)width;
}

// out[to] += norm * blockdiag(W_r) feat[from]   over relation-sorted records {src, dst, etype, norm}
//   forward: from = src, to = dst, wl = w_fwd [R][K = si][B * F],  F = so
//   dX     : from = dst, to = src, wl = w_bwd [R][K = so][B * F],  F = si   (swap = 1)
// threads of a slot: unit u = ks * (B * F / CO) + cg  ->  columns cg*CO .. +CO, input rows ks*KI .. +KI
template <int KI, int CO>
__global__ void __launch_bounds__(512)
fwd_kernel(const float* __restrict__ feat, const int4* __restrict__ pack, int E, const float* __restrict__ wl,
           int K, int F, int B, int t_edge, int swap, float* __restrict__ out) {
  extern __shared__ __align__(16) float sm[];
  const int width = B * F, in_w = B * K, n_cg = width / CO, units = n_cg * (K / KI);
  int4* P_s = reinterpret_cast<int4*>(sm);
  float* X_s = sm + 4 * kChunk;                       // [slots][kDepth][in_w]
  const int slots = blockDim.x / t_edge;
  const int slot = threadIdx.x / t_edge, st = threadIdx.x - slot * t_edge;
  const int e0 = blockIdx.x * kChunk, n = min(E - e0, kChunk);
  for (int i = threadIdx.x; i < n; i += blockDim.x) P_s[i] = __ldg(pack + e0 + i);
  __syncthreads();
  if (slot >= slots) return;
  const int n_my = (n - slot + slots - 1) / slots;    // this slot's edges: slot, slot + slots, ...
  const int4* rec = P_s + slot;
  float* ring = X_s + slot * kDepth * in_w;
  const int pieces = in_w / 4;

  auto gather = [&](int k, int buf) {
    const int4 p = rec[k * slots];
    const float* row = row32(feat, swap ? p.y : p.x, in_w);
    for (int q = st; q < pieces; q += t_edge) cp16(ring + buf * in_w + 4 * q, row + 4 * q);
  };
#pragma unroll
  for (int k = 0; k < kDepth - 1; ++k) {
    if (k < n_my) gather(k, k);
    commit();
  }

  const bool active = st < units;
  const int u = active ? st : 0;
  const int ks = u / n_cg, cg = u - ks * n_cg, j0 = cg * CO, k0 = ks * KI;
  const float* xs = ring + (j0 / F) * K + k0;
  const int vec = (K % 4 == 0 && KI % 4 == 0) ? 4 : (K % 2 == 0 && KI % 2 == 0) ? 2 : 1;
  float* out_j = out + j0;
  const float* wl_j = wl + (size_t)k0 * width + j0;
  float w[KI][CO];
  int cur = -1;
  for (int k = 0; k < n_my; ++k) {
    wait_group<kDepth - 2>();                         // row k has landed (this thread's pieces)
    slot_bar(slot, t_edge);                           // ... everybody's; row k-1 is consumed
    if (k + kDepth - 1 < n_my) gather(k + kDepth - 1, (k + kDepth - 1) % kDepth);
    commit();
    const int4 p = rec[k * slots];
    if (active) {
      if (p.z != cur) {                               // relation run starts: my KI x CO weights
        cur = p.z;
        const float* wr = wl_j + (size_t)(unsigned)cur * ((size_t)K * width);
#pragma unroll
        for (int i = 0; i < KI; ++i) {
          if constexpr (CO == 4) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(wr + (size_t)i * width));
            w[i][0] = t.x; w[i][1] = t.y; w[i][2] = t.z; w[i][3] = t.w;
          } else if constexpr (CO == 2) {
            const float2 t = __ldg(reinterpret_cast<const float2*>(wr + (size_t)i * width));
            w[i][0] = t.x; w[i][1] = t.y;
          } else {
            w[i][0] = __ldg(wr + (size_t)i * width);
          }
        }
      }
      float xv[KI], m[CO];
      lds_n<KI>(xv, xs + (k % kDepth) * in_w, vec);
#pragma unroll
      for (int c = 0; c < CO; ++c) m[c] = 0.f;
#pragma unroll
      for (int i = 0; i < KI; ++i)
#pragma unroll
        for (int c = 0; c < CO; ++c) m[c] = fmaf(xv[i], w[i][c], m[c]);
      red_vec<CO>(const_cast<float*>(row32(out_j, swap ? p.x : p.y, width)), m, __int_as_float(p.w));
    }
  }
}

// dW[r][b][i][o] += norm * x[src][b*si + i] * dagg[dst][b*so + o]     (DGL layout [R][B][si][so])
// unit u = (b * (si/TI) + ti) * (so/TO) + to  owns rows ti*TI .. +TI, columns to*TO .. +TO of block b
template <int TI, int TO>
__global__ void __launch_bounds__(512)
dw_kernel(const float* __restrict__ x, const float* __restrict__ dagg, const int4* __restrict__ pack, int E,
          int SI, int SO, int B, int t_edge, float* __restrict__ dW) {
  extern __shared__ __align__(16) float sm[];
  const int in_w = B * SI, out_w = B * SO, row_w = in_w + out_w;
  const int n_ti = SI / TI, n_to = SO / TO, units = B * n_ti * n_to;
  int4* P_s = reinterpret_cast<int4*>(sm);
  float* R_s = sm + 4 * kChunk;                       // [slots][kDepth][in_w + out_w]: x row then dagg row
  const int slots = blockDim.x / t_edge;
  const int slot = threadIdx.x / t_edge, st = threadIdx.x - slot * t_edge;
  const int e0 = blockIdx.x * kChunk, n = min(E - e0, kChunk);
  for (int i = threadIdx.x; i < n; i += blockDim.x) P_s[i] = __ldg(pack + e0 + i);
  __syncthreads();
  if (slot >= slots) return;
  const int n_my = (n - slot + slots - 1) / slots;
  const int4* rec = P_s + slot;
  float* ring = R_s + slot * kDepth * row_w;
  const int px = in_w / 4, pd = out_w / 4;

  auto gather = [&](int k, int buf) {
    const int4 p = rec[k * slots];
    const float* xr = row32(x, p.x, in_w);
    const float* dr = row32(dagg, p.y, out_w);
    float* dst = ring + buf * row_w;
    for (int q = st; q < px; q += t_edge) cp16(dst + 4 * q, xr + 4 * q);
    for (int q = st; q < pd; q += t_edge) cp16(dst + in_w + 4 * q, dr + 4 * q);
  };
#pragma unroll
  for (int k = 0; k < kDepth - 1; ++k) {
    if (k < n_my) gather(k, k);
    commit();
  }

  const bool active = st < units;
  const int u = active ? st : 0;
  const int to = u % n_to, bt = u / n_to, ti = bt % n_ti, b = bt / n_ti;
  const float* xs = ring + b * SI + ti * TI;
  const float* ds = ring + in_w + b * SO + to * TO;
  const int vx = (SI % 4 == 0 && TI % 4 == 0) ? 4 : (SI % 2 == 0 && TI % 2 == 0) ? 2 : 1;
  const int vd = (SO % 4 == 0 && TO % 4 == 0) ? 4 : (SO % 2 == 0 && TO % 2 == 0) ? 2 : 1;
  float* dW_u = dW + ((size_t)b * SI + ti * TI) * SO + to * TO;
  const size_t KW = (size_t)B * SI * SO;
  float acc[TI][TO];
#pragma unroll
  for (int i = 0; i < TI; ++i)
#pragma unroll
    for (int o = 0; o < TO; ++o) acc[i][o] = 0.f;
  int cur = -1;

  auto flush = [&](int r) {
    float* dst = dW_u + (size_t)(unsigned)r * KW;
#pragma unroll
    for (int i = 0; i < TI; ++i) {
      if (vd >= TO || TO == 1) {
        red_vec<TO>(dst + (size_t)i * SO, acc[i], 1.f);
      } else {
#pragma unroll
        for (int o = 0; o < TO; ++o) atomicAdd(dst + (size_t)i * SO + o, acc[i][o]);
      }
#pragma unroll
      for (int o = 0; o < TO; ++o) acc[i][o] = 0.f;
    }
  };

  for (int k = 0; k < n_my; ++k) {
    wait_group<kDepth - 2>();
    slot_bar(slot, t_edge);
    if (k + kDepth - 1 < n_my) gather(k + kDepth - 1, (k + kDepth - 1) % kDepth);
    commit();
    const int4 p = rec[k * slots];
    if (active) {
      if (p.z != cur) {
        if (cur >= 0) flush(cur);
        cur = p.z;
      }
      const float nv = __int_as_float(p.w);
      float xv[TI], dv[TO];
      lds_n<TI>(xv, xs + (k % kDepth) * row_w, vx);
      lds_n<TO>(dv, ds + (k % kDepth) * row_w, vd);
#pragma unroll
      for (int i = 0; i < TI; ++i) {
        const float xn = nv * xv[i];
#pragma unroll
        for (int o = 0; o < TO; ++o) acc[i][o] = fmaf(xn, dv[o], acc[i][o]);
      }
    }
  }
  if (active && cur >= 0) flush(cur);
}

// ------------------------------------------------------------------------------------------
// host side: choice of the register tile
// ------------------------------------------------------------------------------------------
struct Tile {
  int ki, co;      // rows x columns of a thread's register tile (0 = no tiling fits)
};

// widest column vector dividing `cols`, then the largest instantiated row count dividing `rows` with
// at most 100 registers of tile and at most 512 threads per edge
inline Tile pick_tile(int rows, int cols, int B) {
  static const int kRows[] = {50, 25, 20, 10, 8, 5, 4};
  const int co = cols % 4 == 0 ? 4 : cols % 2 == 0 ? 2 : 1;
  for (int ki : kRows) {
    if (rows % ki != 0 || ki * co > 100) continue;
    if (co == 4 && ki == 50) continue;
    const long long units = (long long)B * cols / co * (rows / ki);
    if (units <= 512) return Tile{ki, co};
  }
  return Tile{0, 0};
}

inline bool eligible(int B, int si, int so) {
  if ((B * si) % 4 != 0 || (B * so) % 4 != 0) return false;            // 16-byte row pieces
  const Tile f = pick_tile(si, so, B), d = pick_tile(so, si, B);
  if (!f.ki || !d.ki) return false;
  // the widest ring (dW: x row + dagg row, kDepth deep, at least one slot) must fit in shared memory
  return sizeof(float) * ((size_t)4 * kChunk + (size_t)kDepth * B * (si + so)) <= 200 * 1024;
}

struct Launch {
  int threads, t_edge, slots;
  size_t smem;
};
inline Launch plan(long long units, int row_floats) {
  Launch l;
  l.t_edge = (int)((units + 31) / 32 * 32);
  l.threads = l.t_edge <= 256 ? 256 : 512;
  l.slots = l.threads / l.t_edge;
  if (l.slots > 8) { l.slots = 8; l.threads = 8 * l.t_edge; }         // named barriers 1..8
  // keep the rings of all slots inside ~96 KB so that two CTAs share an SM
  while (l.slots > 1 && sizeof(float) * (size_t)l.slots * kDepth * row_floats > 96 * 1024) {
    --l.slots;
    l.threads = l.slots * l.t_edge;
  }
  l.smem = sizeof(float) * ((size_t)4 * kChunk + (size_t)l.slots * kDepth * row_floats);
  return l;
}

template <int KI, int CO>
int launch_fwd_t(const float* feat, const void* pack, int E, const float* wl, int K, int F, int B, int swap,
                 float* out, cudaStream_t st) {
  const Launch l = plan((long long)B * F / CO * (K / KI), B * K);
  auto kern = fwd_kernel<KI, CO>;
  KG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem));
  kern<<<kg_div_up(E, kChunk), l.threads, l.smem, st>>>(feat, reinterpret_cast<const int4*>(pack), E, wl, K, F, B,
                                                        l.t_edge, swap, out);
  KG_LAUNCH_OK();
  return KG_OK;
}

template <int TI, int TO>
int launch_dw_t(const float* x, const float* dagg, const void* pack, int E, int SI, int SO, int B, float* dW,
                cudaStream_t st) {
  const Launch l = plan((long long)B * (SI / TI) * (SO / TO), B * (SI + SO));
  auto kern = dw_kernel<TI, TO>;
  KG_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem));
  kern<<<kg_div_up(E, kChunk), l.threads, l.smem, st>>>(x, dagg, reinterpret_cast<const int4*>(pack), E, SI, SO, B,
                                                        l.t_edge, dW);
  KG_LAUNCH_OK();
  return KG_OK;
}

#define KG_TILE_CASE(FN, KI_, CO_, ...) \
  if (t.ki == KI_ && t.co == CO_) return FN<KI_, CO_>(__VA_ARGS__)
#define KG_TILE_DISPATCH(FN, ...)        \
  KG_TILE_CASE(FN, 4, 1, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 4, 2, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 4, 4, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 5, 1, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 5, 2, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 5, 4, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 8, 1, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 8, 2, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 8, 4, __VA_ARGS__);   \
  KG_TILE_CASE(FN, 10, 1, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 10, 2, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 10, 4, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 20, 1, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 20, 2, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 20, 4, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 25, 1, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 25, 2, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 25, 4, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 50, 1, __VA_ARGS__);  \
  KG_TILE_CASE(FN, 50, 2, __VA_ARGS__)

// forward (swap = 0: K = si, F = so, wl = w_fwd) or dX (swap = 1: K = so, F = si, wl = w_bwd)
inline int launch_fwd(const float* feat, const void* pack, int E, const float* wl, int K, int F, int B, int swap,
                      float* out, cudaStream_t st) {
  const Tile t = pick_tile(K, F, B);
  KG_TILE_DISPATCH(launch_fwd_t, feat, pack, E, wl, K, F, B, swap, out, st);
  return kg_fail(KG_ERR_INVALID, "bdd tile: no register tile for %d x %d blocks", K, F);
}

inline int launch_dw(const float* x, const float* dagg, const void* pack, int E, int SI, int SO, int B, float* dW,
                     cudaStream_t st) {
  const Tile t = pick_tile(SI, SO, B);
  KG_TILE_DISPATCH(launch_dw_t, x, dagg, pack, E, SI, SO, B, dW, st);
  return kg_fail(KG_ERR_INVALID, "bdd tile: no register tile for %d x %d blocks", SI, SO);
}

}  // namespace bddtile
