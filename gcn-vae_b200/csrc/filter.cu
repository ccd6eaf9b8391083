// Filter lists for filtered link-prediction metrics and filtered tail generation, built on the device.
// An extension: the reference ranks against all entities (perturb_and_get_rank / sort_and_rank,
// kgvae/utils.py:180-221; calc_mrr, :293-314 - raw only, kgvae/link_predict.py:7) and generates from all entities
// (kgvae/utils.py:245-288).  Host counterpart and test reference: utils.build_filter.
//
// For a query (a, r) the list holds every entity c that forms a known triple with it - (a, r, c) in direction
// KG_FILTER_OBJECT, (c, r, a) in direction KG_FILTER_SUBJECT - ascending and duplicate-free.
//   kg_filter_table   one 64-bit key (a R + r) N + c per known triple, CUB radix sort over the 2 bits(N) + bits(R)
//                     bits in use, duplicates dropped: every query's list is one run of the sorted table
//   kg_filter_count   the run of (a, r) lies between the lower bounds of (a R + r) N and (a R + r + 1) N; the run
//                     lengths are scanned into ptr, and the total is read back once so the caller can size idx
//   kg_filter_gather  one warp per query copies its run's c values into idx
#include <cub/cub.cuh>

#include "common.cuh"

namespace {

constexpr int kThreads = 256;
typedef unsigned long long u64;

int bits_for(int n) {
  int b = 1;
  while (b < 31 && (1ll << b) < (long long)n) ++b;
  return b;
}

__global__ void __launch_bounds__(kThreads)
filter_keys(const int* __restrict__ tri, int T, int N, int R, int direction, u64* __restrict__ keys) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= T) return;
  const int s = __ldg(tri + 3 * (size_t)i), r = __ldg(tri + 3 * (size_t)i + 1), o = __ldg(tri + 3 * (size_t)i + 2);
  const int a = direction == KG_FILTER_OBJECT ? s : o, c = direction == KG_FILTER_OBJECT ? o : s;
  keys[i] = ((u64)a * R + r) * N + c;
}

__device__ __forceinline__ int lower_bound_u64(const u64* __restrict__ t, int lo, int hi, u64 key) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(t + mid) < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// first key of the query's run; false for ids out of range (their list is empty)
__device__ __forceinline__ bool run_base(int a, int r, int N, int R, u64* base) {
  if (a < 0 || a >= N || r < 0 || r >= R) return false;
  *base = ((u64)a * R + r) * N;
  return true;
}

__global__ void __launch_bounds__(kThreads)
filter_count(const u64* __restrict__ table, const int* __restrict__ table_len, int N, int R,
             const int* __restrict__ a, const int* __restrict__ r, int M, long long* __restrict__ cnt) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  const int n = __ldg(table_len);
  u64 base;
  long long c = 0;
  if (run_base(__ldg(a + i), __ldg(r + i), N, R, &base)) {
    const int lo = lower_bound_u64(table, 0, n, base);
    c = lower_bound_u64(table, lo, n, base + N) - lo;
  }
  cnt[i] = c;
}

__global__ void __launch_bounds__(kThreads)
filter_ptr32(const long long* __restrict__ off, int n, int* __restrict__ ptr) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) ptr[i] = (int)off[i];
}

__global__ void __launch_bounds__(kThreads)
filter_gather(const u64* __restrict__ table, const int* __restrict__ table_len, int N, int R,
              const int* __restrict__ a, const int* __restrict__ r, int M, const int* __restrict__ ptr,
              int* __restrict__ idx) {
  const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (m >= M) return;
  const int begin = __ldg(ptr + m), cnt = __ldg(ptr + m + 1) - begin;
  u64 base;
  if (cnt <= 0 || !run_base(__ldg(a + m), __ldg(r + m), N, R, &base)) return;
  const int lo = lower_bound_u64(table, 0, __ldg(table_len), base);     // same value in every lane
  for (int j = lane; j < cnt; j += 32) idx[begin + j] = (int)(__ldg(table + lo + j) - base);
}

size_t table_temp_bytes(int T) {
  size_t a = 0, b = 0;
  cub::DeviceRadixSort::SortKeys((void*)nullptr, a, (u64*)nullptr, (u64*)nullptr, T);
  cub::DeviceSelect::Unique((void*)nullptr, b, (u64*)nullptr, (u64*)nullptr, (int*)nullptr, T);
  return kg_align_up((a > b ? a : b) + 256);
}

size_t count_temp_bytes(int M) {
  size_t a = 0;
  cub::DeviceScan::ExclusiveSum((void*)nullptr, a, (long long*)nullptr, (long long*)nullptr, M + 1);
  return kg_align_up(a + 256);
}

}  // namespace

extern "C" size_t kg_filter_table_workspace_bytes(int n_triples) {
  const int T = n_triples > 0 ? n_triples : 1;
  return 2 * kg_align_up((size_t)T * sizeof(u64)) + table_temp_bytes(T) + 1024;
}

extern "C" int kg_filter_table(const int32_t* triples, int n_triples, int num_nodes, int num_rels, int direction,
                               uint64_t* table, int32_t* table_len, void* workspace, size_t workspace_bytes,
                               void* stream) {
  KG_REQUIRE(n_triples >= 0 && num_nodes > 0 && num_rels > 0, "filter table: bad sizes");
  KG_REQUIRE(direction == KG_FILTER_OBJECT || direction == KG_FILTER_SUBJECT, "filter table: bad direction %d",
             direction);
  const int key_bits = 2 * bits_for(num_nodes) + bits_for(num_rels);
  KG_REQUIRE(key_bits <= 64, "filter table: keys need 2 bits(N) + bits(R) = %d > 64 bits (N = %d, R = %d)", key_bits,
             num_nodes, num_rels);
  cudaStream_t st = kg_stream(stream);
  const int T = n_triples;
  KG_CUDA(cudaMemsetAsync(table_len, 0, sizeof(int32_t), st));
  if (T == 0) return KG_OK;
  KgArena ws(workspace, workspace_bytes);
  u64* keys_in = ws.take<u64>(T);
  u64* keys_out = ws.take<u64>(T);
  size_t temp_bytes = table_temp_bytes(T);
  void* temp = ws.take<char>(temp_bytes);
  if (!workspace || !keys_in || !keys_out || !temp)
    return kg_fail(KG_ERR_WORKSPACE, "filter table: workspace too small (%zu needed)",
                   kg_filter_table_workspace_bytes(T));
  filter_keys<<<kg_div_up(T, kThreads), kThreads, 0, st>>>(triples, T, num_nodes, num_rels, direction, keys_in);
  KG_LAUNCH_OK();
  size_t tb = temp_bytes;
  KG_CUDA(cub::DeviceRadixSort::SortKeys(temp, tb, keys_in, keys_out, T, 0, key_bits, st));
  tb = temp_bytes;
  KG_CUDA(cub::DeviceSelect::Unique(temp, tb, keys_out, reinterpret_cast<u64*>(table), table_len, T, st));
  return KG_OK;
}

extern "C" size_t kg_filter_count_workspace_bytes(int n_queries) {
  const int M = n_queries > 0 ? n_queries : 0;
  return kg_align_up((size_t)(M + 1) * sizeof(long long)) + count_temp_bytes(M) + 1024;
}

extern "C" int kg_filter_count(const uint64_t* table, const int32_t* table_len, int num_nodes, int num_rels,
                               const int32_t* a, const int32_t* r, int n_queries, int32_t* ptr, long long* total,
                               void* workspace, size_t workspace_bytes, void* stream) {
  KG_REQUIRE(n_queries >= 0 && num_nodes > 0 && num_rels > 0 && total != nullptr, "filter count: bad arguments");
  cudaStream_t st = kg_stream(stream);
  const int M = n_queries;
  KgArena ws(workspace, workspace_bytes);
  long long* off = ws.take<long long>(M + 1);
  size_t temp_bytes = count_temp_bytes(M);
  void* temp = ws.take<char>(temp_bytes);
  if (!workspace || !off || !temp)
    return kg_fail(KG_ERR_WORKSPACE, "filter count: workspace too small (%zu needed)",
                   kg_filter_count_workspace_bytes(M));
  KG_CUDA(cudaMemsetAsync(off + M, 0, sizeof(long long), st));
  if (M > 0) {
    filter_count<<<kg_div_up(M, kThreads), kThreads, 0, st>>>(reinterpret_cast<const u64*>(table), table_len,
                                                              num_nodes, num_rels, a, r, M, off);
    KG_LAUNCH_OK();
  }
  size_t tb = temp_bytes;
  KG_CUDA(cub::DeviceScan::ExclusiveSum(temp, tb, off, off, M + 1, st));
  filter_ptr32<<<kg_div_up(M + 1, kThreads), kThreads, 0, st>>>(off, M + 1, ptr);
  KG_LAUNCH_OK();
  // the one read-back: the caller sizes idx with it
  long long sum = 0;
  KG_CUDA(cudaMemcpyAsync(&sum, off + M, sizeof(long long), cudaMemcpyDeviceToHost, st));
  KG_CUDA(cudaStreamSynchronize(st));
  *total = sum;
  if (sum >= (1ll << 31))
    return kg_fail(KG_ERR_INVALID, "filter count: %lld listed entities do not fit int32 offsets", sum);
  return KG_OK;
}

extern "C" int kg_filter_gather(const uint64_t* table, const int32_t* table_len, int num_nodes, int num_rels,
                                const int32_t* a, const int32_t* r, int n_queries, const int32_t* ptr, int32_t* idx,
                                void* stream) {
  KG_REQUIRE(n_queries >= 0 && num_nodes > 0 && num_rels > 0, "filter gather: bad sizes");
  if (n_queries == 0) return KG_OK;
  filter_gather<<<kg_div_up((long long)n_queries * 32, kThreads), kThreads, 0, kg_stream(stream)>>>(
      reinterpret_cast<const u64*>(table), table_len, num_nodes, num_rels, a, r, n_queries, ptr, idx);
  KG_LAUNCH_OK();
  return KG_OK;
}
