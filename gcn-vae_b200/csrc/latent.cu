// a5 / a6 / a7: latent-variable kernels - mean/variance heads with the reparameterised sample,
// the single-sample KL estimate against the mixture-of-Gaussians prior, and the element update of
// one IAF (MADE) pass.  Each replaces a chain of 5-15 ATen elementwise/reduction launches with
// broadcast temporaries ([N, k, h] for the mixture) in the reference.
#include "common.cuh"

static constexpr int kThreads = 256;
static constexpr int kMaxMix = 16;
#define KG_LOG_SQRT_2PI 0.91893853320467274178f

// ------------------------------------------------------------------------------------------
// a5  gaussian_parameters + sample_gaussian   (reference kgvae/utils.py:323-361)
// ------------------------------------------------------------------------------------------
__global__ void reparam_fwd_kernel(const float* __restrict__ h2, const float* __restrict__ eps, int n,
                                   int h, float* __restrict__ zm, float* __restrict__ zv,
                                   float* __restrict__ z) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * h) return;
  int i = (int)(t / h), d = (int)(t % h);
  const float m = h2[(size_t)i * 2 * h + d];
  const float v = kg_softplus(h2[(size_t)i * 2 * h + h + d]) + 1e-8f;   // utils.py:338
  zm[t] = m;
  zv[t] = v;
  z[t] = m + eps[t] * sqrtf(v);                                         // utils.py:359-360
}

__global__ void reparam_bwd_kernel(const float* __restrict__ h2, const float* __restrict__ eps,
                                   const float* __restrict__ zv, const float* __restrict__ dz,
                                   const float* __restrict__ dmean, const float* __restrict__ dvar,
                                   int n, int h, float* __restrict__ dh2) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * h) return;
  int i = (int)(t / h), d = (int)(t % h);
  const float g = dz ? dz[t] : 0.f;
  float gm = g, gv = g * eps[t] * 0.5f / sqrtf(zv[t]);
  if (dmean) gm += dmean[t];
  if (dvar) gv += dvar[t];
  dh2[(size_t)i * 2 * h + d] = gm;
  dh2[(size_t)i * 2 * h + h + d] = gv * kg_sigmoid(h2[(size_t)i * 2 * h + h + d]);
}

extern "C" int kg_reparam_fwd(const float* h2, const float* eps, int n, int h, float* z_mean,
                              float* z_var, float* z, void* stream) {
  KG_REQUIRE(n >= 0 && h > 0, "reparam fwd: bad sizes");
  if (n == 0) return KG_OK;
  reparam_fwd_kernel<<<kg_div_up((long long)n * h, kThreads), kThreads, 0, kg_stream(stream)>>>(
      h2, eps, n, h, z_mean, z_var, z);
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" int kg_reparam_bwd(const float* h2, const float* eps, const float* z_var, const float* dz,
                              const float* dmean, const float* dvar, int n, int h, float* dh2,
                              void* stream) {
  KG_REQUIRE(n >= 0 && h > 0, "reparam bwd: bad sizes");
  if (n == 0) return KG_OK;
  reparam_bwd_kernel<<<kg_div_up((long long)n * h, kThreads), kThreads, 0, kg_stream(stream)>>>(
      h2, eps, z_var, dz, dmean, dvar, n, h, dh2);
  KG_LAUNCH_OK();
  return KG_OK;
}

// ------------------------------------------------------------------------------------------
// a7  KL estimate   (reference kgvae/model.py:82-87, utils.py:364-428)
// prior_ws [3, k, h]: variance, 1/(2 variance), log(sqrt(variance)) of each mixture component
// ------------------------------------------------------------------------------------------
__global__ void prior_prepare_kernel(const float* __restrict__ z_pre, int k, int h,
                                     float* __restrict__ ws) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= k * h) return;
  const float v = kg_softplus(z_pre[(size_t)k * h + t]) + 1e-8f;
  ws[t] = v;
  ws[(size_t)k * h + t] = 1.f / (2.f * v);
  ws[(size_t)2 * k * h + t] = logf(sqrtf(v));
}

// A warp takes kKlWarpRows consecutive rows at a time so that every prior value it fetches
// (3 arrays x k mixtures per column) is applied to several rows.  V = 4: a lane owns float4 column
// groups (h % 4 == 0, 16-byte aligned rows), every load is 128-bit.  The per-element work is kept to
// the essentials: -t^2/(2v) with one approximate division, log(sqrt(v)) = 0.5 log v, and for the
// mixture terms only fma(-(z-m_i)^2, 1/(2 v_i), .): the sum of log(sqrt(v_i)) + log(sqrt(2 pi)) over
// the columns does not depend on the row and is accumulated once per warp.
static constexpr int kKlWarpRows = 4;

template <int KM, int V>
__global__ void __launch_bounds__(128, 4)
kl_mog_fwd_kernel(const float* __restrict__ z, const float* __restrict__ zm,
                  const float* __restrict__ zv, const float* __restrict__ z_pre,
                  const float* __restrict__ ws, int n, int h, int k, float* __restrict__ kl_rows,
                  float* __restrict__ resp, const int* __restrict__ n_valid) {
  const int row0 = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5) * kKlWarpRows;
  const int lane = threadIdx.x & 31;
  // n_valid (device, may be NULL): rows n_valid .. n-1 are padding - kl_rows = 0, nothing else is computed or written
  const int n_rows = n;
  if (n_valid != nullptr) n = min(__ldg(n_valid), n_rows);
  if (row0 >= n) {
    if (lane < kKlWarpRows && row0 + lane < n_rows) kl_rows[row0 + lane] = 0.f;
    return;
  }
  const float* inv2v = ws + (size_t)k * h;
  const float* lsq = ws + (size_t)2 * k * h;
  float a[kKlWarpRows], b[kKlWarpRows][KM], lsum[KM];
#pragma unroll
  for (int i = 0; i < KM; ++i) lsum[i] = 0.f;
#pragma unroll
  for (int q = 0; q < kKlWarpRows; ++q) {
    a[q] = 0.f;
#pragma unroll
    for (int i = 0; i < KM; ++i) b[q][i] = 0.f;
  }
  for (int d = lane * V; d < h; d += 32 * V) {
    float zc[kKlWarpRows][V];
#pragma unroll
    for (int q = 0; q < kKlWarpRows; ++q) {
      const size_t off = (size_t)min(row0 + q, n - 1) * h + d;      // rows past the end repeat the last one (not stored)
      float mc[V], vc[V];
      if (V == 4) {
        const float4 t0 = *reinterpret_cast<const float4*>(z + off), t1 = *reinterpret_cast<const float4*>(zm + off),
                     t2 = *reinterpret_cast<const float4*>(zv + off);
        zc[q][0] = t0.x; zc[q][1] = t0.y; zc[q][V / 2] = t0.z; zc[q][V - 1] = t0.w;
        mc[0] = t1.x; mc[1 % V] = t1.y; mc[V / 2] = t1.z; mc[V - 1] = t1.w;
        vc[0] = t2.x; vc[1 % V] = t2.y; vc[V / 2] = t2.z; vc[V - 1] = t2.w;
      } else {
        zc[q][0] = z[off]; mc[0] = zm[off]; vc[0] = zv[off];
      }
#pragma unroll
      for (int c = 0; c < V; ++c) {
        const float t = zc[q][c] - mc[c];
        a[q] += -__fdividef(t * t, 2.f * vc[c]) - 0.5f * __logf(vc[c]) - KG_LOG_SQRT_2PI;      // utils.py:396
      }
    }
#pragma unroll
    for (int i = 0; i < KM; ++i)
      if (i < k) {
        const size_t po = (size_t)i * h + d;
        float pm[V], iv[V];
        if (V == 4) {
          const float4 t0 = __ldg(reinterpret_cast<const float4*>(z_pre + po)),
                       t1 = __ldg(reinterpret_cast<const float4*>(inv2v + po)),
                       t2 = __ldg(reinterpret_cast<const float4*>(lsq + po));
          pm[0] = t0.x; pm[1 % V] = t0.y; pm[V / 2] = t0.z; pm[V - 1] = t0.w;
          iv[0] = t1.x; iv[1 % V] = t1.y; iv[V / 2] = t1.z; iv[V - 1] = t1.w;
          lsum[i] += (t2.x + t2.y) + (t2.z + t2.w);
        } else {
          pm[0] = __ldg(z_pre + po); iv[0] = __ldg(inv2v + po);
          lsum[i] += __ldg(lsq + po);
        }
#pragma unroll
        for (int q = 0; q < kKlWarpRows; ++q)
#pragma unroll
          for (int c = 0; c < V; ++c) {
            const float u = zc[q][c] - pm[c];
            b[q][i] = fmaf(-(u * u), iv[c], b[q][i]);
          }
      }
  }
  float cst[KM];                                       // sum_d [log(sqrt(v_i)) + log(sqrt(2 pi))]
#pragma unroll
  for (int i = 0; i < KM; ++i) cst[i] = i < k ? kg_warp_sum(lsum[i]) + (float)h * KG_LOG_SQRT_2PI : 0.f;
#pragma unroll
  for (int q = 0; q < kKlWarpRows; ++q) {
    const int row = row0 + q;
    const float aq = kg_warp_sum(a[q]);
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < KM; ++i)
      if (i < k) {
        b[q][i] = kg_warp_sum(b[q][i]) - cst[i];
        mx = fmaxf(mx, b[q][i]);
      }
    float se = 0.f;
#pragma unroll
    for (int i = 0; i < KM; ++i)
      if (i < k) se += expf(b[q][i] - mx);
    const float lse = mx + logf(se);                                        // utils.py:413-415
    if (row < n) {
      if (lane == 0) kl_rows[row] = aq - (lse - logf((float)k));            // utils.py:428, model.py:86
#pragma unroll
      for (int i = 0; i < KM; ++i)
        if (i < k && lane == (i & 31)) resp[(size_t)row * k + i] = expf(b[q][i] - lse);
    } else if (row < n_rows && lane == 0) {
      kl_rows[row] = 0.f;
    }
  }
}

static constexpr int kKlRows = 32;   // rows per CTA in the backward kernel

template <int KM>
__global__ void __launch_bounds__(128, 6)
kl_mog_bwd_kernel(const float* __restrict__ z, const float* __restrict__ zm,
                  const float* __restrict__ zv, const float* __restrict__ z_pre,
                  const float* __restrict__ ws, const float* __restrict__ resp, float scale, int n,
                  int h, int k, const float* __restrict__ coefs, const float* __restrict__ add,
                  float* __restrict__ dz, float* __restrict__ dmean,
                  float* __restrict__ dvar, float* __restrict__ dz_pre, const int* __restrict__ n_valid) {
  const int d = blockIdx.y * blockDim.x + threadIdx.x;
  if (d >= h) return;
  const int r0 = blockIdx.x * kKlRows;
  int r1 = min(n, r0 + kKlRows);
  if (n_valid != nullptr) {
    // rows n_valid .. n-1 are padding: exact zeros in dz / dmean / dvar, nothing added to dz_pre.  The mean's 1/n is
    // formed as the host forms it (a double quotient rounded to float), so valid rows match kg_kl_mog_bwd_fused bitwise
    const int nv = min(__ldg(n_valid), n);
    for (int row = max(r0, nv); row < r1; ++row) {
      const size_t off = (size_t)row * h + d;
      dz[off] = 0.f;
      dmean[off] = 0.f;
      dvar[off] = 0.f;
    }
    r1 = min(r1, nv);
    if (r0 >= r1) return;
    scale = (float)(1.0 / (double)nv);
  }
  // fused form (kg_kl_mog_bwd_fused): the whole gradient of the loss head wrt z in one pass -
  //   dz = coefs[0] * dKL/dz + coefs[1] * add + coefs[2] * z     (add: dz of the DistMult term; z: the regulariser)
  const float c_add = coefs ? __ldg(coefs + 1) : 0.f, c_z = coefs ? __ldg(coefs + 2) : 0.f;
  if (coefs) scale *= __ldg(coefs);
  // per mixture component i and column d, summed over the CTA's rows with r = resp[row, i], u = z - m_i:
  //   gpm = -sum r u / v_i          (gradient wrt the component mean)
  //   gpv = -sum r (u^2 / (2 v_i^2) - 1 / (2 v_i)) = -acc / (2 v_i)   with acc = sum ((r u / v_i) u - r)
  // so the inner loop is eight instructions per (row, component): load r, u, w = u / v_i, q = r w, and the sums.
  float pm[KM], ipv[KM], gpm[KM], acc[KM];
#pragma unroll
  for (int i = 0; i < KM; ++i) {
    pm[i] = i < k ? z_pre[(size_t)i * h + d] : 0.f;
    ipv[i] = i < k ? 1.f / ws[(size_t)i * h + d] : 0.f;
    gpm[i] = 0.f;
    acc[i] = 0.f;
  }
#pragma unroll 2
  for (int row = r0; row < r1; ++row) {
    const size_t off = (size_t)row * h + d;
    const float zc = z[off], v = zv[off];
    const float t = zc - zm[off];
    const float iv = __frcp_rn(v);
    const float tiv = t * iv;
    float gz = -tiv;                         // d/dz log N(z; m, v)
    dmean[off] = scale * tiv;
    dvar[off] = scale * 0.5f * iv * (t * tiv - 1.f);
#pragma unroll
    for (int i = 0; i < KM; ++i)
      if (i < k) {
        const float ri = __ldg(resp + (size_t)row * k + i);
        const float u = zc - pm[i];
        const float q = ri * (u * ipv[i]);   // resp_i * (z - m_i)/v_i
        gz += q;                             // d/dz of -log MoG
        gpm[i] -= q;
        acc[i] += fmaf(q, u, -ri);
      }
    float out = scale * gz;
    if (coefs) out += c_z * zc + (add ? c_add * add[off] : 0.f);
    dz[off] = out;
  }
#pragma unroll
  for (int i = 0; i < KM; ++i)
    if (i < k) {
      atomicAdd(dz_pre + (size_t)i * h + d, scale * gpm[i]);
      atomicAdd(dz_pre + (size_t)(k + i) * h + d,
                scale * (-0.5f * ipv[i] * acc[i]) * kg_sigmoid(z_pre[(size_t)(k + i) * h + d]));
    }
}

static int kl_mog_fwd_impl(const float* z, const float* z_mean, const float* z_var, const float* z_pre, int n, int h,
                           int k, const int* n_valid, float* prior_ws, float* kl_rows, float* resp, void* stream) {
  KG_REQUIRE(n >= 0 && h > 0 && k > 0 && k <= kMaxMix, "kl fwd: need 0 < k <= 16");
  cudaStream_t st = kg_stream(stream);
  prior_prepare_kernel<<<kg_div_up((long long)k * h, kThreads), kThreads, 0, st>>>(z_pre, k, h, prior_ws);
  KG_LAUNCH_OK();
  if (n == 0) return KG_OK;
  const int grid = kg_div_up((long long)kg_div_up(n, kKlWarpRows) * 32, 128);
  const bool vec = h % 4 == 0 && ((reinterpret_cast<uintptr_t>(z) | reinterpret_cast<uintptr_t>(z_mean) |
                                   reinterpret_cast<uintptr_t>(z_var) | reinterpret_cast<uintptr_t>(z_pre) |
                                   reinterpret_cast<uintptr_t>(prior_ws)) & 15) == 0;
#define KG_KL_FWD(KM_)                                                                                          \
  do {                                                                                                          \
    if (vec) kl_mog_fwd_kernel<KM_, 4><<<grid, 128, 0, st>>>(z, z_mean, z_var, z_pre, prior_ws, n, h, k, kl_rows, resp, \
                                                             n_valid);                                          \
    else kl_mog_fwd_kernel<KM_, 1><<<grid, 128, 0, st>>>(z, z_mean, z_var, z_pre, prior_ws, n, h, k, kl_rows, resp,     \
                                                         n_valid);                                              \
  } while (0)
  if (k <= 4) KG_KL_FWD(4);
  else if (k <= 8) KG_KL_FWD(8);
  else if (k <= 12) KG_KL_FWD(12);
  else KG_KL_FWD(16);
#undef KG_KL_FWD
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" int kg_kl_mog_fwd(const float* z, const float* z_mean, const float* z_var,
                             const float* z_pre, int n, int h, int k, float* prior_ws, float* kl_rows,
                             float* resp, void* stream) {
  return kl_mog_fwd_impl(z, z_mean, z_var, z_pre, n, h, k, nullptr, prior_ws, kl_rows, resp, stream);
}

// The same over the first n_valid (device int) of n_rows rows: a sampled subgraph padded to a fixed node budget.
// Rows past n_valid get kl_rows = 0 and cost no work; resp of those rows is not written.
extern "C" int kg_kl_mog_fwd_rows(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                                  int n_rows, int h, int k, const int32_t* n_valid, float* prior_ws, float* kl_rows,
                                  float* resp, void* stream) {
  KG_REQUIRE(n_valid != nullptr, "kl fwd rows: n_valid is required");
  return kl_mog_fwd_impl(z, z_mean, z_var, z_pre, n_rows, h, k, n_valid, prior_ws, kl_rows, resp, stream);
}

// the per-thread mixture arrays are sized by the smallest instantiation that holds k (registers -> occupancy)
static void launch_kl_bwd(dim3 grid, cudaStream_t st, const float* z, const float* zm, const float* zv, const float* z_pre,
                          const float* ws, const float* resp, float scale, int n, int h, int k, const float* coefs,
                          const float* add, float* dz, float* dmean, float* dvar, float* dz_pre,
                          const int* n_valid = nullptr) {
  if (k <= 4) kl_mog_bwd_kernel<4><<<grid, 128, 0, st>>>(z, zm, zv, z_pre, ws, resp, scale, n, h, k, coefs, add, dz, dmean, dvar, dz_pre, n_valid);
  else if (k <= 8) kl_mog_bwd_kernel<8><<<grid, 128, 0, st>>>(z, zm, zv, z_pre, ws, resp, scale, n, h, k, coefs, add, dz, dmean, dvar, dz_pre, n_valid);
  else if (k <= 12) kl_mog_bwd_kernel<12><<<grid, 128, 0, st>>>(z, zm, zv, z_pre, ws, resp, scale, n, h, k, coefs, add, dz, dmean, dvar, dz_pre, n_valid);
  else kl_mog_bwd_kernel<16><<<grid, 128, 0, st>>>(z, zm, zv, z_pre, ws, resp, scale, n, h, k, coefs, add, dz, dmean, dvar, dz_pre, n_valid);
}

extern "C" int kg_kl_mog_bwd(const float* z, const float* z_mean, const float* z_var,
                             const float* z_pre, const float* prior_ws, const float* resp, float scale,
                             int n, int h, int k, float* dz, float* dmean, float* dvar, float* dz_pre,
                             void* stream) {
  KG_REQUIRE(n >= 0 && h > 0 && k > 0 && k <= kMaxMix, "kl bwd: need 0 < k <= 16");
  if (n == 0) return KG_OK;
  dim3 grid(kg_div_up(n, kKlRows), kg_div_up(h, 128));
  launch_kl_bwd(grid, kg_stream(stream), z, z_mean, z_var, z_pre, prior_ws, resp, scale, n, h, k, nullptr, nullptr, dz,
                dmean, dvar, dz_pre);
  KG_LAUNCH_OK();
  return KG_OK;
}

// The same pass producing the COMBINED gradient of the loss head (kgvae/link_predict.py:74-91) wrt z:
//   dz = coefs[0] * scale * dKL/dz + coefs[1] * add + coefs[2] * z;   dmean, dvar, dz_pre scaled by coefs[0] * scale
// coefs: device [3] (upstream gradient times kl_param; times 1 for the DistMult term `add` [n, h], may be NULL;
// times 2 reg_param / (n h) for the regulariser mean(z^2)).
extern "C" int kg_kl_mog_bwd_fused(const float* z, const float* z_mean, const float* z_var,
                                   const float* z_pre, const float* prior_ws, const float* resp, float scale,
                                   int n, int h, int k, const float* coefs, const float* add, float* dz,
                                   float* dmean, float* dvar, float* dz_pre, void* stream) {
  KG_REQUIRE(n >= 0 && h > 0 && k > 0 && k <= kMaxMix, "kl bwd: need 0 < k <= 16");
  KG_REQUIRE(coefs != nullptr, "kl bwd fused: coefs is required");
  if (n == 0) return KG_OK;
  dim3 grid(kg_div_up(n, kKlRows), kg_div_up(h, 128));
  launch_kl_bwd(grid, kg_stream(stream), z, z_mean, z_var, z_pre, prior_ws, resp, scale, n, h, k, coefs, add, dz, dmean,
                dvar, dz_pre);
  KG_LAUNCH_OK();
  return KG_OK;
}

// kg_kl_mog_bwd_fused over the first n_valid (device int) of n_rows rows, scale = 1 / n_valid formed on the device:
// rows n_valid .. n_rows-1 get exact zeros in dz, dmean and dvar and add nothing to dz_pre (CTAs wholly past
// n_valid only write the zeros).
extern "C" int kg_kl_mog_bwd_fused_rows(const float* z, const float* z_mean, const float* z_var, const float* z_pre,
                                        const float* prior_ws, const float* resp, int n_rows, int h, int k,
                                        const int32_t* n_valid, const float* coefs, const float* add, float* dz,
                                        float* dmean, float* dvar, float* dz_pre, void* stream) {
  KG_REQUIRE(n_rows >= 0 && h > 0 && k > 0 && k <= kMaxMix, "kl bwd rows: need 0 < k <= 16");
  KG_REQUIRE(coefs != nullptr && n_valid != nullptr, "kl bwd rows: coefs and n_valid are required");
  if (n_rows == 0) return KG_OK;
  dim3 grid(kg_div_up(n_rows, kKlRows), kg_div_up(h, 128));
  launch_kl_bwd(grid, kg_stream(stream), z, z_mean, z_var, z_pre, prior_ws, resp, 0.f, n_rows, h, k, coefs, add, dz,
                dmean, dvar, dz_pre, n_valid);
  KG_LAUNCH_OK();
  return KG_OK;
}

// ------------------------------------------------------------------------------------------
// a6  IAF element update   (reference kgvae/flow_network.py:91-96)
//
// col_mult[j] = how many times column j occurs in the pass's index list.  0: the column keeps
// x_old.  The reference writes x[:, idx] = z[:, idx] * exp(...) with idx = arange(D) % (D-1) in
// the middle passes, where column 0 is listed twice: the forward value is unchanged, but
// autograd's index_put backward hands the column's gradient to BOTH occurrences, so the
// reference's gradients through that column are doubled.  Reproduced here via the multiplicity.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads)
iaf_update_fwd_kernel(const float* __restrict__ z, const float* __restrict__ net,
                      const float* __restrict__ x_old, const int* __restrict__ col_mult, int n, int d,
                      float* __restrict__ x_new, float* __restrict__ log_det) {
  const int row = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* mu = net + (size_t)row * 2 * d;
  const float* alpha = mu + d;
  float s = 0.f;
  for (int j = lane; j < d; j += 32) {
    const float al = alpha[j];
    s += al;
    const size_t off = (size_t)row * d + j;
    if (__ldg(col_mult + j) == 0) x_new[off] = x_old[off];
    else x_new[off] = z[off] * expf(al + mu[j]);                          // flow_network.py:95
  }
  if (log_det) {
    s = kg_warp_sum(s);
    if (lane == 0) log_det[row] = s;                                       // flow_network.py:96
  }
}

__global__ void iaf_update_bwd_kernel(const float* __restrict__ z, const float* __restrict__ net,
                                      const float* __restrict__ dx_new,
                                      const float* __restrict__ dlog_det,
                                      const int* __restrict__ col_mult, int n, int d,
                                      float* __restrict__ dz, float* __restrict__ dnet,
                                      float* __restrict__ dx_old) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * d) return;
  const int row = (int)(t / d), j = (int)(t % d);
  const int mult = __ldg(col_mult + j);
  const float gl = dlog_det ? dlog_det[row] : 0.f;
  float* dmu = dnet + (size_t)row * 2 * d;
  if (mult == 0) {
    dz[t] = 0.f;
    dmu[j] = 0.f;
    dmu[d + j] = gl;
    dx_old[t] = dx_new[t];
  } else {
    const float g = dx_new[t] * (float)mult;
    const float e = expf(net[(size_t)row * 2 * d + d + j] + net[(size_t)row * 2 * d + j]);
    const float gx = g * z[t] * e;
    dz[t] = g * e;
    dmu[j] = gx;
    dmu[d + j] = gx + gl;
    dx_old[t] = 0.f;
  }
}

extern "C" int kg_iaf_update_fwd(const float* z, const float* net_out, const float* x_old,
                                 const int32_t* col_mult, int n, int d, float* x_new, float* log_det,
                                 void* stream) {
  KG_REQUIRE(n >= 0 && d > 0 && col_mult && x_old, "iaf fwd: bad arguments");
  if (n == 0) return KG_OK;
  iaf_update_fwd_kernel<<<kg_div_up((long long)n * 32, kThreads), kThreads, 0, kg_stream(stream)>>>(
      z, net_out, x_old, col_mult, n, d, x_new, log_det);
  KG_LAUNCH_OK();
  return KG_OK;
}

extern "C" int kg_iaf_update_bwd(const float* z, const float* net_out, const float* dx_new,
                                 const float* dlog_det, const int32_t* col_mult, int n, int d,
                                 float* dz, float* dnet_out, float* dx_old, void* stream) {
  KG_REQUIRE(n >= 0 && d > 0 && col_mult, "iaf bwd: bad arguments");
  if (n == 0) return KG_OK;
  iaf_update_bwd_kernel<<<kg_div_up((long long)n * d, kThreads), kThreads, 0, kg_stream(stream)>>>(
      z, net_out, dx_new, dlog_det, col_mult, n, d, dz, dnet_out, dx_old);
  KG_LAUNCH_OK();
  return KG_OK;
}

__global__ void reverse_columns_kernel(const float* __restrict__ x, int n, int d, float* __restrict__ out) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * d) return;
  const int row = (int)(t / d), j = (int)(t % d);
  out[t] = x[(size_t)row * d + (d - 1 - j)];                               // flow_network.py:26,29
}

extern "C" int kg_reverse_columns(const float* x, int n, int d, float* out, void* stream) {
  KG_REQUIRE(n >= 0 && d > 0, "reverse: bad sizes");
  if (n == 0) return KG_OK;
  reverse_columns_kernel<<<kg_div_up((long long)n * d, kThreads), kThreads, 0, kg_stream(stream)>>>(x, n, d, out);
  KG_LAUNCH_OK();
  return KG_OK;
}
