// a10: all-entity rank evaluation on the 5th-generation tensor cores.
// Replaces utils.perturb_and_get_rank + sort_and_rank (reference kgvae/utils.py:180-221): the
// reference materialises a D x E x V outer-product tensor (11.6 GB per 400-query batch at
// FB15k-237 shape), reduces it to an E x V score matrix, applies sigmoid and fully sorts every
// row to find one position.  Here the M x V score matrix only ever exists as 128 x 256 fp32
// tiles in tensor memory; the epilogue counts, per query, the candidates that beat the target,
// so only int32 ranks[M] reach HBM.
//
// Definition of the score (the "canonical" fp32 value every comparison is decided on):
//   q_i = emb[a_i] * w[r_i]                        (one fp32 multiply per element, utils.py:200)
//   dot(q, e) = butterfly_sum_l( chain_{k = l, l+32, ...} fmaf(q[k], e[k], .) )   (lane l of a warp)
//   score_ij = dot(q_i, emb[j]) + shift            (utils.py:204-207)
//   rank_i = #{j : score_ij > score_i,b_i} + #{j < b_i : score_ij == score_i,b_i}      (SURVEY F4)
// Comparing logits instead of sigmoid(logits) refines the reference's order (sigmoid is monotone),
// so the result always lies inside the reference's tie interval and equals it when the
// reference has no ties.
//
// How the tensor cores are used without giving up the fp32 decision: both operands are split
// into two fp16 terms (x * 2^s = hi + lo, s a per-row power of two), and the tile accumulates
// lo*hi + hi*lo + hi*hi in fp32 (tcgen05.mma kind::f16, operands TMA-staged in 128B-swizzled
// shared memory, accumulators double-buffered in TMEM).  The epilogue treats that value as a
// FILTER: a candidate whose tensor-core score differs from the target's canonical score by more
// than  mu * |q| * |e| + eps  is decided immediately; the few that fall inside the band
// (about 5e-4 of all pairs on Gaussian data, and every exact tie) are re-scored with dot()
// above by the same warp.  mu = 2^-15 is > 10x the worst deviation the split product showed
// against dot() (tests/test_gpu_ops.py::test_rank_filter_margin).
#include "split_pipe.cuh"

using namespace splitpipe;

namespace {

constexpr int SMEM_BYTES = PIPE_SMEM + 1024 + 2 * BN * 8 + 4 * (BN / 32) * 32 * 4;   // + colp_s, amb_s
constexpr float kMu = 3.0517578125e-05f;               // 2^-15
constexpr float kEps = 4.76837158203125e-07f;         // 2^-21

__device__ __forceinline__ float warp_dot(const float* __restrict__ q, const float* __restrict__ e, int h,
                                          int lane) {
  float acc = 0.f;
  for (int k = lane; k < h; k += 32) acc = fmaf(__ldg(q + k), __ldg(e + k), acc);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

// one warp per candidate row n (shard-relative): fp16 split of emb[cand_begin + n] and column record
__global__ void __launch_bounds__(256)
entity_prep(const float* __restrict__ emb, int cand_begin, int n_cand, int n_cols, int h, int Kp,
            __half* __restrict__ bcat, float2* __restrict__ colp) {
  const int n = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (n >= n_cols) return;
  if (n >= n_cand) {                                    // tile overhang: masked out
    if (lane == 0) colp[n] = make_float2(0.f, __int_as_float(0x7fc00000));
    return;
  }
  const float* e = emb + (size_t)(cand_begin + n) * h;
  float amax = 0.f, ss = 0.f;
  for (int k = lane; k < h; k += 32) {
    const float x = __ldg(e + k);
    amax = fmaxf(amax, fabsf(x));
    ss = fmaf(x, x, ss);
  }
  amax = warp_max(amax);
  ss = kg_warp_sum(ss);
  const float s = split_scale(amax);
  __half* row = bcat + (size_t)n * 2 * Kp;
  for (int k = lane; k < Kp; k += 32) {
    if (k < h) split_store(__ldg(e + k), s, row + k, row + Kp + k);
    else { row[k] = __float2half_rn(0.f); row[Kp + k] = __float2half_rn(0.f); }
  }
  if (lane == 0) colp[n] = make_float2(1.f / s, sqrtf(ss) * 1.000002f);
}

// one warp per query: canonical q (fp32), its fp16 split, the target's canonical score and the
// row record {A, B, C, t}:  candidate j is decided by  d = sq*(q.e_j)_tc - A  against  B*|e_j| + C
__global__ void __launch_bounds__(256)
query_prep(const float* __restrict__ emb, const float* __restrict__ w, const int* __restrict__ a,
           const int* __restrict__ r, const int* __restrict__ b, int M, int h, int Kp,
           const float* __restrict__ shift_p, float mu, float* __restrict__ q32, __half* __restrict__ acat,
           float4* __restrict__ rowp, float* __restrict__ sqv) {
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (m >= M) return;
  const float shift = shift_p ? __ldg(shift_p) : 0.f;
  const float* ea = emb + (size_t)__ldg(a + m) * h;
  const float* wr = w + (size_t)__ldg(r + m) * h;
  const float* eb = emb + (size_t)__ldg(b + m) * h;
  float* q = q32 + (size_t)m * h;
  float amax = 0.f, ss = 0.f, acc = 0.f;
  for (int k = lane; k < h; k += 32) {
    const float x = __ldg(ea + k) * __ldg(wr + k);       // utils.py:200
    q[k] = x;
    amax = fmaxf(amax, fabsf(x));
    ss = fmaf(x, x, ss);
    acc = fmaf(x, __ldg(eb + k), acc);                   // same chain as warp_dot
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  amax = warp_max(amax);
  ss = kg_warp_sum(ss);
  const float s = split_scale(amax);
  __half* row = acat + (size_t)m * 2 * Kp;
  for (int k = lane; k < Kp; k += 32) {
    if (k < h) split_store(q[k], s, row + k, row + Kp + k);
    else { row[k] = __float2half_rn(0.f); row[Kp + k] = __float2half_rn(0.f); }
  }
  if (lane == 0) {
    const float t = acc + shift;                         // utils.py:206-207
    rowp[m] = make_float4(s * (t - shift), s * mu * sqrtf(ss) * 1.000002f,
                          s * (kEps * (fabsf(shift) + fabsf(t)) + 1e-37f), t);
    sqv[m] = s;
  }
}

struct RankArgs {
  const float* q32;
  const float* emb;
  const float4* rowp;
  const float2* colp;
  const int* tgt;
  const float* shift;
  int* ranks;
  const float* sqv;      // per-query scale (only read when dump != nullptr)
  float* dump;           // test hook: tensor-core scores [M, n_cand] (nullptr in production)
  int M, h, Kp, cand_begin, n_cand, m_tiles, n_tiles, n_terms;
};

__global__ void __launch_bounds__(THREADS, 1)
rank_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, RankArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const Pipe P = pipe_setup(smem_raw, &tm_a, &tm_b);
  float2* colp_s = reinterpret_cast<float2*>(P.scratch);                       // [2][BN]
  uint32_t* amb_s = reinterpret_cast<uint32_t*>(P.scratch + 2 * BN * 8);       // [4][BN/32][32]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TileMap tmap{p.m_tiles, p.n_tiles, 1, p.Kp / BK, p.Kp / BK};
  const int total = tmap.total();

  if (warp == 0) {
    pipe_producer(P, &tm_a, &tm_b, tmap, p.Kp, p.n_terms);
  } else if (warp == 1) {
    pipe_mma(P, tmap, p.n_terms);
  } else {
    // ---------------------------------------------------------------- epilogue (warps 2..5)
    const int quad = warp & 3;                // TMEM lanes [32*quad, 32*quad + 32)
    const int etid = threadIdx.x - 64;        // 0..127 among the epilogue threads
    const float shift = p.shift ? __ldg(p.shift) : 0.f;
    uint32_t* my_amb = amb_s + (quad * (BN / 32)) * 32 + lane;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const int m0 = (tile / p.n_tiles) * BM, n0 = (tile % p.n_tiles) * BN;
      const int m = m0 + quad * 32 + lane;
      // column records of this tile -> shared memory (double-buffered: one barrier per tile)
      float4* cs4 = reinterpret_cast<float4*>(colp_s + buf * BN);
      cs4[etid] = __ldg(reinterpret_cast<const float4*>(p.colp + n0) + etid);
      float4 rp = make_float4(0.f, __int_as_float(0x7fc00000), 0.f, 0.f);
      int tg = -1;
      if (m < p.M) {
        rp = __ldg(p.rowp + m);
        tg = __ldg(p.tgt + m);
      }
      epi_barrier();
      const uint32_t taddr = epi_acquire(P, it);
      int cnt = 0;
#pragma unroll 1
      for (int c = 0; c < BN / 32; c += 2) {
        uint32_t v0[32], v1[32];
        tmem_ld_32x32b_x32(taddr + c * 32, v0);
        tmem_ld_32x32b_x32(taddr + c * 32 + 32, v1);
        tmem_ld_wait();
        const float4* cp = cs4 + c * 16;
        uint32_t mask0 = 0, mask1 = 0;
#pragma unroll
        for (int j = 0; j < 32; j += 2) {
          const float4 ca = cp[j >> 1], cb = cp[16 + (j >> 1)];   // {1/se, |e|} x 2 columns (broadcast)
          const float d0 = fmaf(__uint_as_float(v0[j]), ca.x, -rp.x), c0 = fmaf(rp.y, ca.y, rp.z);
          const float d1 = fmaf(__uint_as_float(v0[j + 1]), ca.z, -rp.x), c1 = fmaf(rp.y, ca.w, rp.z);
          const float d2 = fmaf(__uint_as_float(v1[j]), cb.x, -rp.x), c2 = fmaf(rp.y, cb.y, rp.z);
          const float d3 = fmaf(__uint_as_float(v1[j + 1]), cb.z, -rp.x), c3 = fmaf(rp.y, cb.w, rp.z);
          cnt += (d0 > c0) + (d1 > c1) + (d2 > c2) + (d3 > c3);
          if (fabsf(d0) <= c0) mask0 |= 1u << j;
          if (fabsf(d1) <= c1) mask0 |= 2u << j;
          if (fabsf(d2) <= c2) mask1 |= 1u << j;
          if (fabsf(d3) <= c3) mask1 |= 2u << j;
        }
        my_amb[c * 32] = mask0;
        my_amb[(c + 1) * 32] = mask1;
        if (p.dump && m < p.M) {                           // test hook: the filter's view of the scores
          const float inv_sq = 1.f / __ldg(p.sqv + m);
          for (int j = 0; j < 64; ++j) {
            const int n = n0 + c * 32 + j;
            const float acc = __uint_as_float(j < 32 ? v0[j & 31] : v1[j & 31]);
            if (n < p.n_cand) p.dump[(size_t)m * p.n_cand + n] = acc * __ldg(&p.colp[n].x) * inv_sq;
          }
        }
      }
      epi_release(P, it);                                  // TMEM buffer may be overwritten
      // undecided pairs: canonical fp32 score, whole warp per pair
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        const uint32_t mine = my_amb[c * 32];
        unsigned any = __ballot_sync(0xffffffffu, mine != 0);
        while (any) {
          const int src = __ffs(any) - 1;
          any &= any - 1;
          uint32_t bits = __shfl_sync(0xffffffffu, mine, src);
          const int mr = __shfl_sync(0xffffffffu, m, src);
          const float t = __shfl_sync(0xffffffffu, rp.w, src);
          const int tgs = __shfl_sync(0xffffffffu, tg, src);
          const float* qrow = p.q32 + (size_t)mr * p.h;
          int extra = 0;
          if (p.h <= 512) {
            float qv[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) qv[i] = lane + 32 * i < p.h ? __ldg(qrow + lane + 32 * i) : 0.f;
            while (bits) {
              const int j = __ffs(bits) - 1;
              bits &= bits - 1;
              const int n = p.cand_begin + n0 + c * 32 + j;
              const float* erow = p.emb + (size_t)n * p.h;
              float ev[16];
#pragma unroll
              for (int i = 0; i < 16; ++i) ev[i] = lane + 32 * i < p.h ? __ldg(erow + lane + 32 * i) : 0.f;
              float acc = 0.f;                              // same chain as warp_dot (zero terms are exact no-ops)
#pragma unroll
              for (int i = 0; i < 16; ++i) acc = fmaf(qv[i], ev[i], acc);
#pragma unroll
              for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
              const float sc = acc + shift;
              extra += (sc > t || (sc == t && n < tgs)) ? 1 : 0;
            }
          } else {
            while (bits) {
              const int j = __ffs(bits) - 1;
              bits &= bits - 1;
              const int n = p.cand_begin + n0 + c * 32 + j;
              const float sc = warp_dot(qrow, p.emb + (size_t)n * p.h, p.h, lane) + shift;
              extra += (sc > t || (sc == t && n < tgs)) ? 1 : 0;
            }
          }
          if (lane == src) cnt += extra;
        }
      }
      if (m < p.M && cnt) atomicAdd(p.ranks + m, cnt);
    }
  }

  pipe_teardown(P);
}

// filtered setting: take back every known-true candidate that was counted (warp per query)
__global__ void __launch_bounds__(256)
filter_correction(const float* __restrict__ q32, const float* __restrict__ emb, const float4* __restrict__ rowp,
                  const int* __restrict__ tgt, const int* __restrict__ filt_ptr,
                  const int* __restrict__ filt_idx, int M, int h, const float* __restrict__ shift_p,
                  int cand_begin, int cand_end, int* __restrict__ ranks) {
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (m >= M) return;
  const float shift = shift_p ? __ldg(shift_p) : 0.f;
  const float t = __ldg(&rowp[m].w);
  const int tid = __ldg(tgt + m);
  int cnt = 0;
  for (int pidx = __ldg(filt_ptr + m); pidx < __ldg(filt_ptr + m + 1); ++pidx) {
    const int j = __ldg(filt_idx + pidx);
    if (j == tid || j < cand_begin || j >= cand_end) continue;
    const float s = warp_dot(q32 + (size_t)m * h, emb + (size_t)j * h, h, lane) + shift;
    cnt += (s > t || (s == t && j < tid)) ? 1 : 0;
  }
  if (lane == 0 && cnt) atomicSub(ranks + m, cnt);
}

// ------------------------------------------------------------------------------------------
// top-k tails: the same score tiles with a top-k epilogue (reference kgvae/utils.py:245-288, `generate`:
// argmax tail per query; k = 1 there).  Each epilogue thread owns one query row of the tile and keeps the
// KK = k + 1 best tensor-core scores of the tile's 256 candidates in registers; they go to a
// [M, n_tiles, KK] candidate list.  A finish kernel re-scores every listed candidate with the canonical
// fp32 dot product and keeps the k best by (score desc, entity id asc); a tile whose (k+1)-th listed score
// could still reach the k-th exact score (within the filter's error band) is re-scanned completely, so
// the result does not depend on the tensor-core rounding.
// Filtered generation (FILT, an extension): each query's listed entities (ascending CSR) are scored -inf in the
// tile epilogue, so every tile's list holds its best UNLISTED candidates and the error-band argument above holds
// for the unlisted entities; the re-scan of a tile skips the listed ones too.  FILT = false is the unfiltered
// kernel unchanged (the filter fields sit behind the ones it reads).
// Sharded generation: the candidates are entities [cand_begin, cand_begin + n_cand).  The tiles and their lists
// use shard-relative ids n; the filter lists hold global ids (compared against cand_begin + n) and the finish pass
// writes global ids.  The band's |e| maximum is taken over the shard's own candidates, so the argument holds per
// launch.  Every score is the canonical one, so merging the shards' lists by (score desc, id asc) is exact.
// ------------------------------------------------------------------------------------------
struct TopkArgs {
  const float2* colp;
  const float* sqv;
  float* cand_v;
  int* cand_i;
  int M, Kp, n_cand, m_tiles, n_tiles, n_terms;
  const int* filt_ptr;   // FILT only
  const int* filt_idx;
  int cand_begin;
};

// first position in v[lo, hi) whose value is >= key
__device__ __forceinline__ int lower_bound_i32(const int* __restrict__ v, int lo, int hi, int key) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(v + mid) < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

template <int KK>
__device__ __forceinline__ void topk_insert(float (&bv)[KK], int (&bi)[KK], float v, int n) {
  if (!(v > bv[KK - 1])) return;
  bv[KK - 1] = v;
  bi[KK - 1] = n;
#pragma unroll
  for (int i = KK - 1; i > 0; --i) {
    if (bv[i] > bv[i - 1]) {
      const float tv = bv[i]; bv[i] = bv[i - 1]; bv[i - 1] = tv;
      const int ti = bi[i]; bi[i] = bi[i - 1]; bi[i - 1] = ti;
    }
  }
}

template <int KK, bool FILT>
__global__ void __launch_bounds__(THREADS, 1)
topk_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, TopkArgs p) {
  extern __shared__ uint8_t smem_raw[];
  const Pipe P = pipe_setup(smem_raw, &tm_a, &tm_b);
  float2* colp_s = reinterpret_cast<float2*>(P.scratch);                       // [2][BN]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TileMap tmap{p.m_tiles, p.n_tiles, 1, p.Kp / BK, p.Kp / BK};
  const int total = tmap.total();
  if (warp == 0) {
    pipe_producer(P, &tm_a, &tm_b, tmap, p.Kp, p.n_terms);
  } else if (warp == 1) {
    pipe_mma(P, tmap, p.n_terms);
  } else {
    const int quad = warp & 3, etid = threadIdx.x - 64;
    int it = 0;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const int n_tile = tile % p.n_tiles, m0 = (tile / p.n_tiles) * BM, n0 = n_tile * BN;
      const int m = m0 + quad * 32 + lane;
      float4* cs4 = reinterpret_cast<float4*>(colp_s + buf * BN);
      cs4[etid] = __ldg(reinterpret_cast<const float4*>(p.colp + n0) + etid);
      const float inv_sq = m < p.M ? 1.f / __ldg(p.sqv + m) : 0.f;
      epi_barrier();
      const uint32_t taddr = epi_acquire(P, it);
      float bv[KK];
      int bi[KK];
#pragma unroll
      for (int i = 0; i < KK; ++i) { bv[i] = -INFINITY; bi[i] = -1; }
      const float2* cs = colp_s + buf * BN;
      int fc = 0, fe = 0;            // FILT: cursor into this row's list, at its first id >= cand_begin + n0
      if constexpr (FILT) {
        if (m < p.M) {
          fe = __ldg(p.filt_ptr + m + 1);
          fc = lower_bound_i32(p.filt_idx, __ldg(p.filt_ptr + m), fe, p.cand_begin + n0);
        }
      }
#pragma unroll 1
      for (int c = 0; c < BN / 32; ++c) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + c * 32, v);
        uint32_t listed = 0;           // FILT: bit j = entity cand_begin + n0 + 32 c + j is listed
        if constexpr (FILT) {
          for (; fc < fe; ++fc) {
            const int j = __ldg(p.filt_idx + fc) - (p.cand_begin + n0 + c * 32);
            if (j >= 32) break;
            if (j >= 0) listed |= 1u << j;
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float2 cp = cs[c * 32 + j];                                    // {1 / s_e, |e|}: broadcast
          const int n = n0 + c * 32 + j;
          float val = n < p.n_cand ? __uint_as_float(v[j]) * cp.x * inv_sq : -INFINITY;
          if constexpr (FILT) {
            if ((listed >> j) & 1u) val = -INFINITY;
          }
          topk_insert<KK>(bv, bi, val, n);
        }
      }
      epi_release(P, it);
      if (m < p.M) {
        float* ov = p.cand_v + ((size_t)m * p.n_tiles + n_tile) * KK;
        int* oi = p.cand_i + ((size_t)m * p.n_tiles + n_tile) * KK;
#pragma unroll
        for (int i = 0; i < KK; ++i) { ov[i] = bv[i]; oi[i] = bi[i]; }
      }
    }
  }
  pipe_teardown(P);
}

// max_j |e_j| over the candidate records (one block)
__global__ void __launch_bounds__(256)
colp_max_kernel(const float2* __restrict__ colp, int n_cand, float* __restrict__ out) {
  __shared__ float red[8];
  float m = 0.f;
  for (int i = threadIdx.x; i < n_cand; i += 256) m = fmaxf(m, __ldg(&colp[i].y));
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
    out[0] = m;
  }
}

constexpr int kTopkMax = 10;

// one warp per query; every lane keeps the same sorted list (scores are warp-uniform after the butterfly sum).
// emb points at the shard's first row (entity cand_begin): the ids n below are shard-relative, the output global.
// FILT: the tiles' candidate lists hold no listed entity (the epilogue scored them -inf), the re-scan skips them.
template <bool FILT>
__global__ void __launch_bounds__(256)
topk_finish_kernel(const float* __restrict__ q32, const float* __restrict__ emb, const float4* __restrict__ rowp,
                   const float* __restrict__ sqv, const float* __restrict__ cand_v, const int* __restrict__ cand_i,
                   const float* __restrict__ emax_p, int M, int h, int cand_begin, int n_cand, int n_tiles, int KK,
                   int k, const float* __restrict__ shift_p, int* __restrict__ out_idx, float* __restrict__ out_score,
                   const int* __restrict__ filt_ptr, const int* __restrict__ filt_idx) {
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (m >= M) return;
  const float shift = shift_p ? __ldg(shift_p) : 0.f;
  const float* q = q32 + (size_t)m * h;
  float ts[kTopkMax];
  int ti[kTopkMax];
#pragma unroll
  for (int i = 0; i < kTopkMax; ++i) { ts[i] = -INFINITY; ti[i] = 0x7fffffff; }
  auto offer = [&](float sc, int n) {           // order: score descending, entity id ascending; no duplicates
#pragma unroll
    for (int i = 0; i < kTopkMax; ++i)
      if (ti[i] == n) return;
    if (!(sc > ts[kTopkMax - 1] || (sc == ts[kTopkMax - 1] && n < ti[kTopkMax - 1]))) return;
    ts[kTopkMax - 1] = sc;
    ti[kTopkMax - 1] = n;
#pragma unroll
    for (int i = kTopkMax - 1; i > 0; --i) {
      if (ts[i] > ts[i - 1] || (ts[i] == ts[i - 1] && ti[i] < ti[i - 1])) {
        const float tv = ts[i]; ts[i] = ts[i - 1]; ts[i - 1] = tv;
        const int tn = ti[i]; ti[i] = ti[i - 1]; ti[i - 1] = tn;
      }
    }
  };
  const float* cv = cand_v + (size_t)m * n_tiles * KK;
  const int* ci = cand_i + (size_t)m * n_tiles * KK;
  for (int t = 0; t < n_tiles; ++t)
    for (int i = 0; i < KK; ++i) {
      const int n = __ldg(ci + t * KK + i);
      if (n < 0) continue;
      offer(warp_dot(q, emb + (size_t)n * h, h, lane) + shift, n);
    }
  // error band of a tensor-core score in real units: mu |q| |e| (+ eps terms), |q| recovered from the row record
  const float4 rp = __ldg(rowp + m);
  const float s = __ldg(sqv + m);
  const float band = (rp.y / s) * __ldg(emax_p) * 1.01f + 4.f * kEps * (fabsf(shift) + fabsf(ts[0] - shift)) + 1e-30f;
  for (int t = 0; t < n_tiles; ++t) {
    const float v_last = __ldg(cv + t * KK + KK - 1);        // the best score NOT kept is <= this one
    if (!(v_last + shift + band >= ts[k - 1])) continue;
    const int n_end = min(n_cand, (t + 1) * BN);
    int fc = 0, fe = 0, nx = 0x7fffffff;        // FILT: the row's next listed id >= n, shard-relative (warp-uniform)
    if constexpr (FILT) {
      fe = __ldg(filt_ptr + m + 1);
      fc = lower_bound_i32(filt_idx, __ldg(filt_ptr + m), fe, cand_begin + t * BN);
      nx = fc < fe ? __ldg(filt_idx + fc) - cand_begin : 0x7fffffff;
    }
    for (int n = t * BN; n < n_end; ++n) {
      if constexpr (FILT) {
        bool listed = false;
        while (nx <= n) {
          listed |= nx == n;
          ++fc;
          nx = fc < fe ? __ldg(filt_idx + fc) - cand_begin : 0x7fffffff;
        }
        if (listed) continue;
      }
      offer(warp_dot(q, emb + (size_t)n * h, h, lane) + shift, n);
    }
  }
  if (lane == 0)
    for (int i = 0; i < k; ++i) {
      out_idx[(size_t)m * k + i] = ti[i] == 0x7fffffff ? -1 : cand_begin + ti[i];
      out_score[(size_t)m * k + i] = ts[i];
    }
}

struct Layout {
  size_t q32, acat, bcat, rowp, colp, sqv, total;
  int Kp, n_tiles, m_tiles;
};

Layout layout(int M, int n_cand, int h) {
  Layout L;
  L.Kp = kg_div_up(h, BK) * BK;
  L.m_tiles = kg_div_up(M, BM);
  L.n_tiles = kg_div_up(n_cand, BN);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += kg_align_up(bytes, 1024); return o; };
  L.q32 = take((size_t)M * h * sizeof(float));
  L.acat = take((size_t)M * 2 * L.Kp * sizeof(__half));
  L.bcat = take((size_t)(n_cand > 0 ? n_cand : 1) * 2 * L.Kp * sizeof(__half));
  L.rowp = take((size_t)M * sizeof(float4));
  L.colp = take((size_t)(L.n_tiles > 0 ? L.n_tiles : 1) * BN * sizeof(float2));
  L.sqv = take((size_t)M * sizeof(float));
  L.total = off;
  return L;
}

}  // namespace

extern "C" size_t kg_distmult_rank_workspace_bytes(int n_queries, int n_candidates, int h) {
  if (n_queries <= 0 || h <= 0) return 1024;
  return layout(n_queries, n_candidates > 0 ? n_candidates : 0, h).total + 1024;
}

extern "C" int kg_distmult_rank(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                                const int32_t* b, int n_queries, int n_entities, int h, const float* shift,
                                int cand_begin, int cand_end, const int32_t* filt_ptr,
                                const int32_t* filt_idx, void* workspace, size_t workspace_bytes,
                                int32_t* ranks, float* tc_scores, void* stream) {
  KG_REQUIRE(n_queries >= 0 && n_entities > 0 && h > 0, "rank: bad sizes");
  KG_REQUIRE(0 <= cand_begin && cand_begin <= cand_end && cand_end <= n_entities, "rank: bad candidate shard");
  KG_REQUIRE((filt_ptr == nullptr) == (filt_idx == nullptr), "rank: filter needs both ptr and idx");
  cudaStream_t st = kg_stream(stream);
  const int M = n_queries, n_cand = cand_end - cand_begin;
  if (M == 0) return KG_OK;
  KG_CUDA(cudaMemsetAsync(ranks, 0, sizeof(int) * M, st));
  const Layout L = layout(M, n_cand, h);
  uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023;
  if (!workspace || base + L.total > reinterpret_cast<uintptr_t>(workspace) + workspace_bytes)
    return kg_fail(KG_ERR_WORKSPACE, "rank: workspace too small (%zu needed)", L.total + 1024);
  char* ws = reinterpret_cast<char*>(base);
  float* q32 = reinterpret_cast<float*>(ws + L.q32);
  __half* acat = reinterpret_cast<__half*>(ws + L.acat);
  __half* bcat = reinterpret_cast<__half*>(ws + L.bcat);
  float4* rowp = reinterpret_cast<float4*>(ws + L.rowp);
  float2* colp = reinterpret_cast<float2*>(ws + L.colp);
  float* sqv = reinterpret_cast<float*>(ws + L.sqv);

  // single-product mode: the tensor-core score IS the decision (no band; only exact ties are re-scored)
  const int n_terms = tc05::tc_terms();
  query_prep<<<kg_div_up((long long)M * 32, 256), 256, 0, st>>>(emb, w, a, r, b, M, h, L.Kp, shift,
                                                               n_terms == 3 ? kMu : 0.f, q32, acat, rowp, sqv);
  KG_LAUNCH_OK();
  if (n_cand == 0) return KG_OK;
  const int n_cols = L.n_tiles * BN;
  entity_prep<<<kg_div_up((long long)n_cols * 32, 256), 256, 0, st>>>(emb, cand_begin, n_cand, n_cols, h, L.Kp, bcat, colp);
  KG_LAUNCH_OK();

  CUtensorMap tm_a, tm_b;
  const uint64_t row_bytes = (uint64_t)2 * L.Kp * sizeof(__half);
  int rc = make_tensor_map_2d_b16(&tm_a, acat, M, 2 * L.Kp, row_bytes, BM);
  if (rc != KG_OK) return rc;
  rc = make_tensor_map_2d_b16(&tm_b, bcat, n_cand, 2 * L.Kp, row_bytes, BN);
  if (rc != KG_OK) return rc;

  if (kg_attr_needed(1))
    KG_CUDA(cudaFuncSetAttribute(rank_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  RankArgs args;
  args.q32 = q32; args.emb = emb; args.rowp = rowp; args.colp = colp; args.tgt = b; args.shift = shift;
  args.ranks = ranks; args.sqv = sqv; args.dump = tc_scores;
  args.M = M; args.h = h; args.Kp = L.Kp; args.cand_begin = cand_begin; args.n_cand = n_cand;
  args.m_tiles = L.m_tiles; args.n_tiles = L.n_tiles; args.n_terms = n_terms;
  const int total = L.m_tiles * L.n_tiles;
  const int grid = total < kg_sm_count() ? total : kg_sm_count();
  rank_tc_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(tm_a, tm_b, args);
  KG_LAUNCH_OK();
  if (filt_ptr) {
    filter_correction<<<kg_div_up((long long)M * 32, 256), 256, 0, st>>>(
        q32, emb, rowp, b, filt_ptr, filt_idx, M, h, shift, cand_begin, cand_end, ranks);
    KG_LAUNCH_OK();
  }
  return KG_OK;
}

static int topk_kk(int k) { return k <= 1 ? 2 : (k <= 3 ? 4 : kTopkMax + 1); }

extern "C" size_t kg_distmult_topk_workspace_bytes(int n_queries, int n_entities, int h, int k) {
  if (n_queries <= 0 || h <= 0 || n_entities <= 0) return 1024;
  const Layout L = layout(n_queries, n_entities, h);
  const size_t cand = (size_t)n_queries * L.n_tiles * topk_kk(k);
  return L.total + kg_align_up(cand * sizeof(float), 1024) + kg_align_up(cand * sizeof(int), 1024) + 2048;
}

// fill a [M, k] result with -1 / -inf (an empty shard)
__global__ void __launch_bounds__(256)
topk_empty_kernel(long long n, int* __restrict__ out_idx, float* __restrict__ out_score) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) { out_idx[i] = -1; out_score[i] = -INFINITY; }
}

// out_idx [n_queries, k] int32 (global entity ids, best first; -1 when fewer than k eligible entities),
// out_score [n_queries, k] fp32 canonical scores (+ shift): the k highest-scored tails of each query (a_i, r_i)
// among the entities [cand_begin, cand_end), or among those of them not in the query's filter list
// (filt_ptr != nullptr).
extern "C" int kg_distmult_topk_shard(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                                      int n_queries, int n_entities, int h, const float* shift, int k,
                                      int cand_begin, int cand_end, const int32_t* filt_ptr,
                                      const int32_t* filt_idx, void* workspace, size_t workspace_bytes,
                                      int32_t* out_idx, float* out_score, void* stream) {
  KG_REQUIRE(n_queries >= 0 && n_entities > 0 && h > 0, "topk: bad sizes");
  KG_REQUIRE(k >= 1 && k <= kTopkMax, "topk: k must be in 1..10");
  KG_REQUIRE(0 <= cand_begin && cand_begin <= cand_end && cand_end <= n_entities, "topk: bad candidate shard");
  KG_REQUIRE((filt_ptr == nullptr) == (filt_idx == nullptr), "topk: filter needs both ptr and idx");
  cudaStream_t st = kg_stream(stream);
  const int M = n_queries, n_cand = cand_end - cand_begin;
  if (M == 0) return KG_OK;
  if (n_cand == 0) {
    const long long n = (long long)M * k;
    topk_empty_kernel<<<kg_div_up(n, 256), 256, 0, st>>>(n, out_idx, out_score);
    KG_LAUNCH_OK();
    return KG_OK;
  }
  const Layout L = layout(M, n_cand, h);
  const int KK = topk_kk(k);
  const size_t cand = (size_t)M * L.n_tiles * KK;
  uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023;
  const size_t need = L.total + kg_align_up(cand * sizeof(float), 1024) + kg_align_up(cand * sizeof(int), 1024) + 1024;
  if (!workspace || base + need > reinterpret_cast<uintptr_t>(workspace) + workspace_bytes)
    return kg_fail(KG_ERR_WORKSPACE, "topk: workspace too small (%zu needed)", need + 1024);
  char* ws = reinterpret_cast<char*>(base);
  float* q32 = reinterpret_cast<float*>(ws + L.q32);
  __half* acat = reinterpret_cast<__half*>(ws + L.acat);
  __half* bcat = reinterpret_cast<__half*>(ws + L.bcat);
  float4* rowp = reinterpret_cast<float4*>(ws + L.rowp);
  float2* colp = reinterpret_cast<float2*>(ws + L.colp);
  float* sqv = reinterpret_cast<float*>(ws + L.sqv);
  float* cand_v = reinterpret_cast<float*>(ws + L.total);
  int* cand_i = reinterpret_cast<int*>(ws + L.total + kg_align_up(cand * sizeof(float), 1024));
  float* emax = reinterpret_cast<float*>(ws + L.total + kg_align_up(cand * sizeof(float), 1024) +
                                         kg_align_up(cand * sizeof(int), 1024));

  const int n_terms = tc05::tc_terms();
  // the target slot of the row record is unused here: hand the subject in as a dummy target
  query_prep<<<kg_div_up((long long)M * 32, 256), 256, 0, st>>>(emb, w, a, r, a, M, h, L.Kp, shift, kMu, q32, acat, rowp, sqv);
  KG_LAUNCH_OK();
  const int n_cols = L.n_tiles * BN;
  entity_prep<<<kg_div_up((long long)n_cols * 32, 256), 256, 0, st>>>(emb, cand_begin, n_cand, n_cols, h, L.Kp, bcat, colp);
  KG_LAUNCH_OK();
  colp_max_kernel<<<1, 256, 0, st>>>(colp, n_cand, emax);
  KG_LAUNCH_OK();
  CUtensorMap tm_a, tm_b;
  const uint64_t row_bytes = (uint64_t)2 * L.Kp * sizeof(__half);
  int rc = make_tensor_map_2d_b16(&tm_a, acat, M, 2 * L.Kp, row_bytes, BM);
  if (rc != KG_OK) return rc;
  rc = make_tensor_map_2d_b16(&tm_b, bcat, n_cand, 2 * L.Kp, row_bytes, BN);
  if (rc != KG_OK) return rc;
  TopkArgs args;
  args.colp = colp; args.sqv = sqv; args.cand_v = cand_v; args.cand_i = cand_i;
  args.M = M; args.Kp = L.Kp; args.n_cand = n_cand; args.m_tiles = L.m_tiles; args.n_tiles = L.n_tiles;
  args.n_terms = n_terms;
  args.filt_ptr = filt_ptr; args.filt_idx = filt_idx; args.cand_begin = cand_begin;
  const int total = L.m_tiles * L.n_tiles;
  const int grid = total < kg_sm_count() ? total : kg_sm_count();
#define KG_TOPK_LAUNCH(KK_, FILT_, SLOT_)                                                                       \
  do {                                                                                                          \
    if (kg_attr_needed(SLOT_))                                                                                  \
      KG_CUDA(cudaFuncSetAttribute(topk_tc_kernel<KK_, FILT_>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                   SMEM_BYTES));                                                                \
    topk_tc_kernel<KK_, FILT_><<<grid, THREADS, SMEM_BYTES, st>>>(tm_a, tm_b, args);                            \
  } while (0)
  const int fgrid = kg_div_up((long long)M * 32, 256);
  const float* emb_c = emb + (size_t)cand_begin * h;
  if (filt_ptr == nullptr) {
    if (KK == 2) KG_TOPK_LAUNCH(2, false, 2);
    else if (KK == 4) KG_TOPK_LAUNCH(4, false, 3);
    else KG_TOPK_LAUNCH(kTopkMax + 1, false, 4);
    KG_LAUNCH_OK();
    topk_finish_kernel<false><<<fgrid, 256, 0, st>>>(q32, emb_c, rowp, sqv, cand_v, cand_i, emax, M, h, cand_begin,
                                                     n_cand, L.n_tiles, KK, k, shift, out_idx, out_score, nullptr,
                                                     nullptr);
  } else {
    if (KK == 2) KG_TOPK_LAUNCH(2, true, 6);
    else if (KK == 4) KG_TOPK_LAUNCH(4, true, 7);
    else KG_TOPK_LAUNCH(kTopkMax + 1, true, 8);
    KG_LAUNCH_OK();
    topk_finish_kernel<true><<<fgrid, 256, 0, st>>>(q32, emb_c, rowp, sqv, cand_v, cand_i, emax, M, h, cand_begin,
                                                    n_cand, L.n_tiles, KK, k, shift, out_idx, out_score, filt_ptr,
                                                    filt_idx);
  }
#undef KG_TOPK_LAUNCH
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" int kg_distmult_topk(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                                int n_queries, int n_entities, int h, const float* shift, int k,
                                void* workspace, size_t workspace_bytes, int32_t* out_idx, float* out_score,
                                void* stream) {
  return kg_distmult_topk_shard(emb, w, a, r, n_queries, n_entities, h, shift, k, 0, n_entities, nullptr, nullptr,
                                workspace, workspace_bytes, out_idx, out_score, stream);
}

extern "C" int kg_distmult_topk_filtered(const float* emb, const float* w, const int32_t* a, const int32_t* r,
                                         int n_queries, int n_entities, int h, const float* shift, int k,
                                         const int32_t* filt_ptr, const int32_t* filt_idx, void* workspace,
                                         size_t workspace_bytes, int32_t* out_idx, float* out_score, void* stream) {
  KG_REQUIRE(filt_ptr != nullptr && filt_idx != nullptr, "topk filtered: needs both filt_ptr and filt_idx");
  return kg_distmult_topk_shard(emb, w, a, r, n_queries, n_entities, h, shift, k, 0, n_entities, filt_ptr, filt_idx,
                                workspace, workspace_bytes, out_idx, out_score, stream);
}
