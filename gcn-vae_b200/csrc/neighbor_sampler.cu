// Neighbourhood-expansion edge sampler (kgvae/utils.py:33-76, --edge-sampler neighbor) on the device.
//
// The procedure (tests/neighbor_mirror.py restates it in numpy and is its specification): per pick i, J = 8 caller
// words w[i, 0..7] drive
//   1. a vertex draw v ~ cnt * seen (or ~ [cnt > 0] when that sums to 0):  r = (w0 W) >> 32, v = first entity whose
//      inclusive prefix sum of the weights exceeds r;
//   2. up to R = 6 rejection tries j = (w_t deg[v]) >> 32 on v's adjacency list, taking the first entry whose edge is
//      not picked (the reference's own loop, truncated);
//   3. if none succeeded, the k-th unpicked entry of v's list with k = (w7 cnt[v]) >> 32 - the conditional law of the
//      reference's rejection loop, since cnt[v] is always the number of unpicked entries of v;
//   4. picked[e] = 1, cnt[v] -= 1, cnt[other] -= 1 (a self-loop loses 2), seen[v] = seen[other] = 1.
//
// Picks within one sample are sequential; samples are independent.  One launch draws a bank of samples, one warp per
// sample, with the sample's state - cnt, the seen and picked bits, and two 32-ary sum trees over the entities (one for
// cnt * seen, one for [cnt > 0]) - in shared memory when it fits the device's per-block limit, else in a per-warp
// slab of the workspace.  The adjacency CSR is read-only and shared by all samples (L2-resident at FB15k-237).
// Output depends only on (graph, words): no atomics, no inter-sample communication.
#include "common.cuh"

namespace {

constexpr int kWords = KG_NEIGHBOR_WORDS;
constexpr int kTries = KG_NEIGHBOR_TRIES;
constexpr int kMaxLevels = 6;                         // 32^6 = 2^30 > any admissible entity count
constexpr unsigned kFull = 0xffffffffu;
constexpr size_t kBudget = size_t(1) << 30;           // words + bank + global slabs of one launch
constexpr int kStaticSmem = 1024;                     // headroom for the kernel's static shared level tables
static_assert(kWords >= kTries + 2 && kWords * 4 <= 32, "a pick's words must fit one lane group of 8");

// Word offsets of one sample's state.  cnt [N] first, then the seen bits, the picked bits, the levels 1..top of the
// cnt * seen tree (A), the levels of the [cnt > 0] tree (B).  Level l has size[l] = ceil(size[l-1] / 32) entries and
// the top level has at most 32; size[0] = N are the leaves, computed from cnt and seen instead of stored.
struct Layout {
  int levels;
  int size[kMaxLevels + 1];
  int off_a[kMaxLevels + 1], off_b[kMaxLevels + 1];
  int seen_off, picked_off, zero_end, words;
};

size_t align4(size_t x) { return (x + 3) & ~size_t(3); }

Layout make_layout(int N, int T) {
  Layout L{};
  L.size[0] = N;
  int lv = 0;
  while (L.size[lv] > 32) {
    L.size[lv + 1] = (L.size[lv] + 31) / 32;
    ++lv;
  }
  L.levels = lv;
  size_t off = align4(N);
  L.seen_off = (int)off;
  off += align4((N + 31) / 32);
  L.picked_off = (int)off;
  off += align4(((size_t)T + 31) / 32);
  for (int l = 1; l <= lv; ++l) L.off_a[l] = (int)off, off += align4(L.size[l]);
  L.zero_end = (int)off;                             // seen, picked and tree A start at zero
  for (int l = 1; l <= lv; ++l) L.off_b[l] = (int)off, off += align4(L.size[l]);
  L.words = (int)off;
  return L;
}

__device__ __forceinline__ uint32_t warp_scan(uint32_t x, int lane) {
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(kFull, x, o);
    if (lane >= o) x += y;
  }
  return x;
}

// One level of the descent: lanes hold the 32 child weights x; returns the first child whose inclusive prefix
// exceeds r and lowers r by the weight of the children before it.
__device__ __forceinline__ int pick_child(uint32_t x, uint32_t& r, int lane) {
  const uint32_t incl = warp_scan(x, lane);
  const uint32_t hit = __ballot_sync(kFull, incl > r);
  const int c = hit ? __ffs(hit) - 1 : 31;            // hit != 0 while the trees match cnt and seen
  r -= __shfl_sync(kFull, incl - x, c);
  return c;
}

__device__ __forceinline__ bool bit(const uint32_t* bits, int i) { return (bits[i >> 5] >> (i & 31)) & 1u; }

__device__ __forceinline__ uint32_t mul_hi(uint32_t w, uint32_t n) { return (uint32_t)(((uint64_t)w * n) >> 32); }

template <bool kShared>
__global__ void __launch_bounds__(32) neighbor_sample_kernel(const int* __restrict__ adj_ptr,
                                                             const int2* __restrict__ adj, const Layout L, int B,
                                                             int n_samples, const uint32_t* __restrict__ words,
                                                             int* __restrict__ picks, int* __restrict__ fallbacks,
                                                             uint32_t* __restrict__ slabs) {
  extern __shared__ uint32_t smem[];
  // the level tables are indexed at run time: shared copies keep them out of local memory
  __shared__ int size_[kMaxLevels + 1], off_a[kMaxLevels + 1], off_b[kMaxLevels + 1];
  uint32_t* st = kShared ? smem : slabs + (size_t)blockIdx.x * L.words;
  const int lane = threadIdx.x;
  const int N = L.size[0];
  if (lane <= kMaxLevels) {
    size_[lane] = L.size[lane];
    off_a[lane] = L.off_a[lane];
    off_b[lane] = L.off_b[lane];
  }
  __syncwarp();
  int* cnt = reinterpret_cast<int*>(st);
  uint32_t* seen = st + L.seen_off;
  uint32_t* picked = st + L.picked_off;

  for (int s = blockIdx.x; s < n_samples; s += gridDim.x) {
    // ---- state: cnt = deg, nothing seen or picked, tree A = 0, tree B = number of entities with edges
    for (int i = L.seen_off + lane; i < L.zero_end; i += 32) st[i] = 0;
    uint32_t WA = 0, WB = 0;                          // tree totals, identical in every lane
    for (int base = 0; base < N; base += 32) {
      const int v = base + lane;
      const int d = v < N ? __ldg(adj_ptr + v + 1) - __ldg(adj_ptr + v) : 0;
      if (v < N) cnt[v] = d;
      const uint32_t has = __ballot_sync(kFull, d > 0);
      WB += __popc(has);
      if (L.levels > 0 && lane == 0) st[off_b[1] + (base >> 5)] = __popc(has);
    }
    for (int l = 2; l <= L.levels; ++l) {
      __syncwarp();
      for (int base = 0; base < size_[l - 1]; base += 32) {
        const int c = base + lane;
        const int x = kg_warp_sum_int(c < size_[l - 1] ? (int)st[off_b[l - 1] + c] : 0);
        if (lane == 0) st[off_b[l] + (base >> 5)] = x;
      }
    }
    __syncwarp();

    // ---- picks; the words of 4 picks (one 128-byte line) are loaded one group ahead
    const uint32_t* w = words + (size_t)s * B * kWords;
    const long long nw = (long long)B * kWords;
    uint32_t cur = lane < nw ? __ldcs(w + lane) : 0u;
    uint32_t nxt = 32 + lane < nw ? __ldcs(w + 32 + lane) : 0u;
    int* out = picks + (size_t)s * B;
    int mine = 0, n_fallback = 0;
    for (int i = 0; i < B; ++i) {
      const int q = i & 3;
      if (q == 0 && i > 0) {
        cur = nxt;
        const long long k = (long long)(i + 4) * kWords + lane;
        nxt = k < nw ? __ldcs(w + k) : 0u;
      }
      // 1. vertex draw down the tree in use
      const bool use_a = WA > 0;
      uint32_t r = mul_hi(__shfl_sync(kFull, cur, q * kWords), use_a ? WA : WB);
      int idx = 0;
      for (int l = L.levels; l >= 1; --l) {
        const int c = idx * 32 + lane;
        const uint32_t x = c < size_[l] ? st[(use_a ? off_a[l] : off_b[l]) + c] : 0u;
        idx = idx * 32 + pick_child(x, r, lane);
      }
      {
        const int u = idx * 32 + lane;
        uint32_t x = 0;
        if (u < N) {
          const int cu = cnt[u];
          x = use_a ? ((seen[idx] >> lane) & 1u ? (uint32_t)cu : 0u) : (cu > 0 ? 1u : 0u);
        }
        idx = idx * 32 + pick_child(x, r, lane);
      }
      const int v = idx < N ? idx : N - 1;
      const int beg = __ldg(adj_ptr + v), deg = __ldg(adj_ptr + v + 1) - beg;
      const int cv = cnt[v];

      // 2. rejection tries, all R at once: lane t evaluates try t + 1, the first success wins
      const uint32_t wt = __shfl_sync(kFull, cur, q * kWords + 1 + (lane < kTries ? lane : 0));
      const uint32_t wk = __shfl_sync(kFull, cur, q * kWords + 1 + kTries);
      int2 ent = make_int2(0, 0);
      bool ok = false;
      if (lane < kTries) {
        ent = __ldg(adj + beg + mul_hi(wt, (uint32_t)deg));
        ok = !bit(picked, ent.x);
      }
      const uint32_t okb = __ballot_sync(kFull, ok);
      int e, other;
      if (okb) {
        const int t = __ffs(okb) - 1;
        e = __shfl_sync(kFull, ent.x, t);
        other = __shfl_sync(kFull, ent.y, t);
      } else {
        // 3. the k-th unpicked entry in list order, 32 entries per step
        ++n_fallback;
        uint32_t k = mul_hi(wk, (uint32_t)cv);
        e = -1, other = 0;
        for (int b0 = 0; b0 < deg; b0 += 32) {
          const int j = b0 + lane;
          bool un = false;
          if (j < deg) {
            ent = __ldg(adj + beg + j);
            un = !bit(picked, ent.x);
          }
          const uint32_t ub = __ballot_sync(kFull, un);
          const uint32_t pc = __popc(ub);
          if (k < pc) {
            const uint32_t before = __popc(ub & ((1u << lane) - 1u));
            const int t = __ffs(__ballot_sync(kFull, un && before == k)) - 1;
            e = __shfl_sync(kFull, ent.x, t);
            other = __shfl_sync(kFull, ent.y, t);
            break;
          }
          k -= pc;
        }
        if (e < 0) {                                 // unreachable while cnt[v] counts v's unpicked entries
          e = __shfl_sync(kFull, ent.x, 0);
          other = __shfl_sync(kFull, ent.y, 0);
        }
      }

      // 4. record: leaf weights of v and other change, the deltas walk up both trees (lane l owns level l)
      const bool sv = bit(seen, v), so = bit(seen, other);
      const int co = cnt[other];
      int cv_new, co_new, da_v, db_v, da_o = 0, db_o = 0;
      if (other == v) {
        cv_new = co_new = cv - 2;
      } else {
        cv_new = cv - 1;
        co_new = co - 1;
        da_o = co_new - (so ? co : 0);
        db_o = (co_new > 0) - (co > 0);
      }
      da_v = cv_new - (sv ? cv : 0);
      db_v = (cv_new > 0) - (cv > 0);
      WA += (uint32_t)(da_v + da_o);
      WB += (uint32_t)(db_v + db_o);
      __syncwarp();
      if (lane == 0) {
        picked[e >> 5] |= 1u << (e & 31);
        cnt[v] = cv_new;
        seen[v >> 5] |= 1u << (v & 31);
        if (other != v) {
          cnt[other] = co_new;
          seen[other >> 5] |= 1u << (other & 31);
        }
      } else if (lane <= L.levels) {
        const int sh = 5 * lane;
        uint32_t* ta = st + off_a[lane];
        uint32_t* tb = st + off_b[lane];
        ta[v >> sh] += (uint32_t)da_v;
        tb[v >> sh] += (uint32_t)db_v;
        ta[other >> sh] += (uint32_t)da_o;
        tb[other >> sh] += (uint32_t)db_o;
      }
      __syncwarp();
      if (lane == (i & 31)) mine = e;
      if ((i & 31) == 31 || i == B - 1) {
        if (lane <= (i & 31)) out[i - (i & 31) + lane] = mine;
      }
    }
    if (fallbacks != nullptr && lane == 0) fallbacks[s] = n_fallback;
    __syncwarp();
  }
}

struct Plan {
  Layout L;
  bool shared;
  size_t state_bytes;
  int resident;                                       // warps (= samples) resident in one wave
};

int make_plan(int N, int T, Plan& p) {
  p.L = make_layout(N, T);
  p.state_bytes = (size_t)p.L.words * 4;
  int dev = 0, optin = 0, sms = kg_sm_count();
  KG_CUDA(cudaGetDevice(&dev));
  KG_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
  const int dyn_max = optin - kStaticSmem;
  p.shared = p.state_bytes <= (size_t)dyn_max;
  int per_sm = 0;
  if (p.shared) {
    if (kg_attr_needed(5))
      KG_CUDA(cudaFuncSetAttribute(neighbor_sample_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn_max));
    KG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, neighbor_sample_kernel<true>, 32, p.state_bytes));
  } else {
    KG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, neighbor_sample_kernel<false>, 32, 0));
  }
  p.resident = (per_sm > 0 ? per_sm : 1) * sms;
  return KG_OK;
}

}  // namespace

extern "C" int kg_neighbor_sample_plan(int num_nodes, int n_triples, int sample_size, int* samples_per_launch,
                                       size_t* workspace_bytes) {
  KG_REQUIRE(num_nodes > 0 && num_nodes < (1 << 30) && n_triples > 0 && n_triples < (1 << 30),
             "neighbor_sample: need 0 < num_nodes, n_triples < 2^30");
  KG_REQUIRE(sample_size >= 1 && sample_size <= n_triples, "neighbor_sample: sample_size must be in 1 .. n_triples");
  KG_REQUIRE(samples_per_launch && workspace_bytes, "neighbor_sample_plan: null output");
  Plan p;
  int rc = make_plan(num_nodes, n_triples, p);
  if (rc != KG_OK) return rc;
  // one sample costs its words and its bank row, plus its slab when the state lives in global memory
  const size_t per = (size_t)sample_size * (kWords + 1) * 4 + (p.shared ? 0 : p.state_bytes);
  size_t k = kBudget / per;
  if (k > (size_t)p.resident) k = p.resident;
  if (k < 1) k = 1;
  *samples_per_launch = (int)k;
  *workspace_bytes = p.shared ? 0 : k * p.state_bytes;
  return KG_OK;
}

extern "C" int kg_neighbor_sample(const int32_t* adj_ptr, const int32_t* adj, int num_nodes, int n_triples,
                                  int sample_size, int n_samples, const uint32_t* words, int32_t* picks,
                                  int32_t* fallbacks, void* workspace, size_t workspace_bytes, void* stream) {
  KG_REQUIRE(num_nodes > 0 && num_nodes < (1 << 30) && n_triples > 0 && n_triples < (1 << 30),
             "neighbor_sample: need 0 < num_nodes, n_triples < 2^30");
  KG_REQUIRE(sample_size >= 1 && sample_size <= n_triples, "neighbor_sample: sample_size must be in 1 .. n_triples");
  KG_REQUIRE(n_samples >= 0, "neighbor_sample: bad sample count");
  KG_REQUIRE(adj_ptr && adj && words && picks, "neighbor_sample: null argument");
  if (n_samples == 0) return KG_OK;
  Plan p;
  int rc = make_plan(num_nodes, n_triples, p);
  if (rc != KG_OK) return rc;
  int grid = n_samples < p.resident ? n_samples : p.resident;
  cudaStream_t st = kg_stream(stream);
  if (p.shared) {
    neighbor_sample_kernel<true><<<grid, 32, p.state_bytes, st>>>(adj_ptr, reinterpret_cast<const int2*>(adj), p.L,
                                                                   sample_size, n_samples, words, picks, fallbacks,
                                                                   nullptr);
  } else {
    const size_t fit = workspace ? workspace_bytes / p.state_bytes : 0;
    if (fit < 1) return kg_fail(KG_ERR_WORKSPACE, "neighbor_sample: workspace too small for one sample's state");
    if ((size_t)grid > fit) grid = (int)fit;
    neighbor_sample_kernel<false><<<grid, 32, 0, st>>>(adj_ptr, reinterpret_cast<const int2*>(adj), p.L, sample_size,
                                                       n_samples, words, picks, fallbacks,
                                                       reinterpret_cast<uint32_t*>(workspace));
  }
  KG_LAUNCH_OK();
  return KG_OK;
}
