// a1-a3: the per-batch graph construction the reference does on the host with pandas and Python
// loops (etpgt/train/dataloader.py:107-202; scripts/pipeline/run_full_pipeline.py:120-166), moved
// onto the device.  Integer work, bit-exact against oracle/graph_ref.py.
//
//   etpgt_item_graph_build     one-off: lookup structure over the stored co-occurrence edge list
//                              (rows keyed by item_i, sorted by item_j, payload = stored row index)
//   etpgt_session_subgraphs_*  per batch: context = all but the last of the (last max_len) events,
//                              nodes = sorted unique context items, edges = stored edges with both
//                              ends in the context, in stored order and direction (+ the
//                              pipeline's symmetrise / self-loop-if-empty rules), PyG collate layout
//   etpgt_sample_negatives     counter-based Philox4x32-10 rejection sampler
//
// One warp per session.  The reference scans the whole 738k-row edge frame twice per session;
// here a session with k nodes does k^2 binary searches in the rows of its own items.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;
constexpr int kWarpsPerCta = kThreads / 32;
constexpr int kMaxCtx = 64;  // context items per session held in shared memory (max_len - 1 <= 63)

// ---------------------------------------------------------------------------- item graph
__global__ void edge_keys_kernel(const int64_t* __restrict__ item_i, const int64_t* __restrict__ item_j, int64_t n,
                                 int64_t num_items, uint64_t* __restrict__ keys, int32_t* __restrict__ iota) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    keys[e] = (uint64_t)item_i[e] * (uint64_t)num_items + (uint64_t)item_j[e];
    iota[e] = (int32_t)e;
  }
}

__global__ void split_keys_kernel(const uint64_t* __restrict__ sorted, int64_t n, int64_t num_items,
                                  int32_t* __restrict__ gcol, int32_t* __restrict__ gptr) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p <= n; p += (int64_t)gridDim.x * blockDim.x) {
    if (p < n) gcol[p] = (int32_t)(sorted[p] % (uint64_t)num_items);
    const int64_t prev = p == 0 ? -1 : (int64_t)(sorted[p - 1] / (uint64_t)num_items);
    int64_t cur = p == n ? num_items : (int64_t)(sorted[p] / (uint64_t)num_items);
    if (cur > num_items) cur = num_items;
    for (int64_t r = prev + 1; r <= cur; ++r) gptr[r] = (int32_t)p;
  }
}

size_t sort64_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)n, 0, 64);
  return bytes;
}

// ---------------------------------------------------------------------------- session warp

struct SessionCtx {
  int64_t nodes[kMaxCtx];  // sorted unique context items
  int64_t raw[kMaxCtx];
  int first[kMaxCtx];
};

// Loads the context of session s (all but the last of its last max_len events), and leaves the
// sorted unique items in ctx.nodes.  Returns the node count (warp-uniform).
__device__ __forceinline__ int load_context(SessionCtx& ctx, const int64_t* __restrict__ sess_ptr,
                                            const int64_t* __restrict__ sess_items, int64_t s, int max_len,
                                            int lane, int64_t* target) {
  const int64_t begin = sess_ptr[s], end = sess_ptr[s + 1];
  int64_t len = end - begin;
  int64_t first_ev = begin;
  if (len > max_len) { first_ev = end - max_len; len = max_len; }
  const int n = len > 0 ? (int)(len - 1) : 0;  // context length
  if (target != nullptr && lane == 0) *target = len > 0 ? sess_items[end - 1] : 0;
  for (int t = lane; t < n; t += 32) ctx.raw[t] = sess_items[first_ev + t];
  __syncwarp();
  // first[t] = no equal item earlier in the context
  for (int t = lane; t < n; t += 32) {
    const int64_t v = ctx.raw[t];
    int is_first = 1;
    for (int u = 0; u < t; ++u) is_first &= ctx.raw[u] != v;
    ctx.first[t] = is_first;
  }
  __syncwarp();
  int k_local = 0;
  for (int t = lane; t < n; t += 32) {
    if (!ctx.first[t]) continue;
    const int64_t v = ctx.raw[t];
    int rank = 0;
    for (int u = 0; u < n; ++u) rank += ctx.first[u] && ctx.raw[u] < v;
    ctx.nodes[rank] = v;
    ++k_local;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) k_local += __shfl_xor_sync(0xffffffffu, k_local, off);
  __syncwarp();
  return k_local;
}

// position of `want` in the sorted row [lo, hi) of gcol, or -1
__device__ __forceinline__ int find_in_row(const int32_t* __restrict__ gcol, int lo, int hi, int32_t want) {
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int32_t v = gcol[mid];
    if (v < want) lo = mid + 1; else hi = mid;
  }
  return (lo < hi || false) ? lo : -1;
}

__device__ __forceinline__ int lookup_edge(const int32_t* __restrict__ gptr, const int32_t* __restrict__ gcol,
                                           int64_t a, int64_t b) {
  int lo = gptr[a];
  const int hi0 = gptr[a + 1];
  int hi = hi0;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (gcol[mid] < (int32_t)b) lo = mid + 1; else hi = mid;
  }
  return (lo < hi0 && gcol[lo] == (int32_t)b) ? lo : -1;
}

template <bool FILL>
__global__ void __launch_bounds__(kThreads)
session_subgraph_kernel(const int32_t* __restrict__ gptr, const int32_t* __restrict__ gcol,
                        const int32_t* __restrict__ gidx, const int64_t* __restrict__ sess_ptr,
                        const int64_t* __restrict__ sess_items, const int64_t* __restrict__ session_ids,
                        int64_t num_sessions, int max_len, int symmetrize,
                        int self_loop_if_empty, int32_t* __restrict__ node_cnt, int32_t* __restrict__ edge_cnt,
                        const int32_t* __restrict__ node_ptr, const int32_t* __restrict__ edge_ptr,
                        int64_t* __restrict__ x, int64_t* __restrict__ batch, int64_t* __restrict__ edge_src,
                        int64_t* __restrict__ edge_dst, int64_t* __restrict__ target,
                        int32_t* __restrict__ tmp_idx, int32_t* __restrict__ tmp_pair) {
  __shared__ SessionCtx ctxs[kWarpsPerCta];
  const int lane = threadIdx.x & 31;
  SessionCtx& ctx = ctxs[threadIdx.x >> 5];
  const int64_t s = (blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5;
  if (s >= num_sessions) return;  // warp-uniform
  int64_t* tgt = FILL ? target + s : nullptr;
  const int64_t sid = session_ids != nullptr ? session_ids[s] : s;
  const int k = load_context(ctx, sess_ptr, sess_items, sid, max_len, lane, tgt);
  const int pairs = k * k;
  const int nbase = FILL ? node_ptr[s] : 0;
  const int ebase = FILL ? edge_ptr[s] : 0;
  if (FILL) {
    for (int t = lane; t < k; t += 32) { x[nbase + t] = ctx.nodes[t]; batch[nbase + t] = s; }
  }
  // stored edges with both ends in the context: ordered pairs (a -> b) of nodes
  int found = 0;
  for (int p0 = 0; p0 < pairs; p0 += 32) {
    const int p = p0 + lane;
    int hit = -1;
    if (p < pairs) hit = lookup_edge(gptr, gcol, ctx.nodes[p / k], ctx.nodes[p % k]);
    const unsigned votes = __ballot_sync(0xffffffffu, hit >= 0);
    if (FILL && hit >= 0) {
      const int slot = found + __popc(votes & ((1u << lane) - 1u));
      tmp_idx[ebase + slot] = gidx[hit];
      tmp_pair[ebase + slot] = p;
    }
    found += __popc(votes);
  }
  const bool loops = self_loop_if_empty && found == 0;
  const int total = loops ? k : (symmetrize ? 2 * found : found);
  if (!FILL) {
    if (lane == 0) { node_cnt[s] = k; edge_cnt[s] = total; }
    return;
  }
  __syncwarp();
  if (loops) {
    for (int t = lane; t < k; t += 32) { edge_src[ebase + t] = nbase + t; edge_dst[ebase + t] = nbase + t; }
    return;
  }
  // stored (CSV) order inside the session: rank of each hit by its stored row index
  for (int h = lane; h < found; h += 32) {
    const int mine = tmp_idx[ebase + h];
    int rank = 0;
    for (int u = 0; u < found; ++u) rank += tmp_idx[ebase + u] < mine;
    const int p = tmp_pair[ebase + h];
    const int64_t a = nbase + p / k, b = nbase + p % k;
    edge_src[ebase + rank] = a;
    edge_dst[ebase + rank] = b;
    if (symmetrize) { edge_src[ebase + found + rank] = b; edge_dst[ebase + found + rank] = a; }
  }
}

__global__ void set_zero_kernel(int32_t* p) { *p = 0; }

// ---------------------------------------------------------------------------- Philox sampler
// (philox4x32_10 lives in common.cuh)

// One thread per (session, slot).  Stream definition: oracle/graph_ref.sample_negatives.
__global__ void __launch_bounds__(kThreads)
sample_negatives_kernel(uint64_t seed, uint32_t step, int64_t session_base, const int64_t* __restrict__ sess_ptr,
                        const int64_t* __restrict__ sess_items, const int64_t* __restrict__ session_ids,
                        int64_t num_sessions, int max_len,
                        int64_t num_items, int num_neg, int64_t* __restrict__ out) {
  const int64_t t = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  if (t >= num_sessions * num_neg) return;
  const int64_t s = t / num_neg;
  const uint32_t slot = (uint32_t)(t % num_neg);
  const int64_t sid = session_ids != nullptr ? session_ids[s] : s;
  const int64_t end = sess_ptr[sid + 1];
  int64_t begin = sess_ptr[sid];
  if (end - begin > max_len) begin = end - max_len;
  const uint64_t gsid = (uint64_t)(session_ids != nullptr ? sid : session_base + s);
  const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  const uint64_t span = (uint64_t)(num_items - 1);
  for (uint32_t attempt = 0;; ++attempt) {
    uint32_t c[4] = {(uint32_t)gsid, slot, attempt >> 2, step};
    philox4x32_10(c, k0, k1);
    const uint32_t word = c[attempt & 3];
    const int64_t cand = 1 + (int64_t)(((uint64_t)word * span) >> 32);
    bool member = false;
    for (int64_t i = begin; i < end; ++i) member |= sess_items[i] == cand;
    if (!member) { out[t] = cand; return; }
  }
}

// Shared negative pool: draw j uses Philox4x32-10 with key (seed lo, seed hi) and counter (j >> 1, "POOL", 0,
// step), 64-bit word c[2 (j & 1)] | c[2 (j & 1) + 1] << 32.  The second counter word keeps the stream apart from
// sample_negatives (whose second word is a slot < 64).  r = floor(u W / 2^64) picks the item i with
// cum[i] <= r < cum[i + 1]: zero-weight items are never drawn.  Stream definition: sample_item_pool in
// tests/shared_pool_ref.py.
__device__ __forceinline__ int64_t upper_bound_i64(const int64_t* __restrict__ a, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] <= x) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(kThreads)
sample_item_pool_kernel(const int64_t* __restrict__ cum, int64_t num_items, int64_t m, uint64_t seed, uint32_t step,
                        uint64_t* __restrict__ out) {
  const int64_t j = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  if (j >= m) return;
  uint32_t c[4] = {(uint32_t)(j >> 1), 0x504F4F4Cu /* "POOL" */, 0u, step};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  const int h = 2 * (int)(j & 1);
  const uint64_t u = (uint64_t)c[h] | ((uint64_t)c[h + 1] << 32);
  const uint64_t r = __umul64hi(u, (uint64_t)cum[num_items]);
  int64_t i = upper_bound_i64(cum, num_items + 1, (int64_t)r) - 1;
  if (i > num_items - 1) i = num_items - 1;  // only when W = 0, which the caller rules out
  out[j] = (uint64_t)i;
}

// log_q[j] = log(M w / W) of the sorted pool, in fp64
__global__ void __launch_bounds__(kThreads)
pool_log_q_kernel(const int64_t* __restrict__ cum, int64_t num_items, const int64_t* __restrict__ pool, int64_t m,
                  float* __restrict__ log_q) {
  const int64_t j = blockIdx.x * (int64_t)kThreads + threadIdx.x;
  if (j >= m) return;
  const int64_t i = pool[j];
  const double w = (double)(cum[i + 1] - cum[i]);
  log_q[j] = (float)log((double)m * w / (double)cum[num_items]);
}

size_t sort_keys64_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortKeys(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr, (int)n, 0, 64);
  return bytes;
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_sample_item_pool_workspace_bytes(int64_t num_sampled) {
  const int64_t m = num_sampled > 0 ? num_sampled : 1;
  return align_up(m * sizeof(uint64_t)) + align_up(sort_keys64_temp_bytes(m)) + 256;
}

extern "C" int etpgt_sample_item_pool(const int64_t* cum, int64_t num_items, int64_t num_sampled, uint64_t seed,
                                      uint32_t step, int64_t* pool_ids, float* log_q, void* ws, size_t ws_bytes,
                                      etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_items >= 1 && num_items < (int64_t(1) << 62), "sample_item_pool: num_items must be >= 1 (got %lld)",
                (long long)num_items);
  ETPGT_REQUIRE(num_sampled >= 1 && num_sampled < (int64_t(1) << 31),
                "sample_item_pool: num_sampled must be in [1, 2^31) (got %lld)", (long long)num_sampled);
  ETPGT_REQUIRE(cum != nullptr, "sample_item_pool: cum is required");
  ETPGT_REQUIRE(pool_ids != nullptr && log_q != nullptr, "sample_item_pool: pool_ids and log_q are required");
  const size_t need = etpgt_sample_item_pool_workspace_bytes(num_sampled);
  if (ws == nullptr || ws_bytes < need) {
    set_error("sample_item_pool: workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return ETPGT_EWORKSPACE;
  }
  Workspace w(ws, ws_bytes);
  uint64_t* drawn = w.take<uint64_t>(num_sampled);
  size_t temp_bytes = sort_keys64_temp_bytes(num_sampled);
  void* temp = w.take<char>(temp_bytes);
  const unsigned grid = (unsigned)((num_sampled + kThreads - 1) / kThreads);
  sample_item_pool_kernel<<<grid, kThreads, 0, stream>>>(cum, num_items, num_sampled, seed, step, drawn);
  ETPGT_CHECK_LAUNCH("sample_item_pool");
  int bits = 1;
  while (bits < 63 && (int64_t(1) << bits) < num_items) ++bits;
  cudaError_t err = cub::DeviceRadixSort::SortKeys(temp, temp_bytes, drawn, reinterpret_cast<uint64_t*>(pool_ids),
                                                   (int)num_sampled, 0, bits, stream);
  if (err != cudaSuccess) { set_error("sample_item_pool sort: %s", cudaGetErrorString(err)); return ETPGT_ECUDA; }
  count_launch(4);
  pool_log_q_kernel<<<grid, kThreads, 0, stream>>>(cum, num_items, pool_ids, num_sampled, log_q);
  ETPGT_CHECK_LAUNCH("sample_item_pool_log_q");
  return ETPGT_OK;
}

extern "C" size_t etpgt_item_graph_workspace_bytes(int64_t num_edges) {
  const int64_t e = num_edges > 0 ? num_edges : 1;
  return 2 * align_up(e * sizeof(uint64_t)) + align_up(e * sizeof(int32_t)) + align_up(sort64_temp_bytes(e)) + 256;
}

extern "C" int etpgt_item_graph_build(const int64_t* item_i, const int64_t* item_j, int64_t num_edges,
                                      int64_t num_items, int32_t* gptr, int32_t* gcol, int32_t* gidx, void* ws,
                                      size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_edges >= 0 && num_items > 0 && num_edges < (int64_t(1) << 31) && num_items < (int64_t(1) << 31),
                "item_graph_build: bad sizes");
  if (ws_bytes < etpgt_item_graph_workspace_bytes(num_edges)) {
    set_error("item_graph_build: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  Workspace w(ws, ws_bytes);
  const int64_t e = num_edges;
  uint64_t* keys = w.take<uint64_t>(e > 0 ? e : 1);
  uint64_t* sorted = w.take<uint64_t>(e > 0 ? e : 1);
  int32_t* iota = w.take<int32_t>(e > 0 ? e : 1);
  const int grid = grid_for(e + 1, kThreads, 8);
  if (e > 0) {
    size_t temp_bytes = sort64_temp_bytes(e);
    void* temp = w.take<char>(temp_bytes);
    edge_keys_kernel<<<grid, kThreads, 0, stream>>>(item_i, item_j, e, num_items, keys, iota);
    ETPGT_CHECK_LAUNCH("edge_keys");
    int bits = 1;
    while (bits < 64 && (uint64_t(1) << bits) < (uint64_t)num_items * (uint64_t)num_items) ++bits;
    cudaError_t err = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, sorted, iota, gidx, (int)e, 0, bits, stream);
    if (err != cudaSuccess) { set_error("item_graph sort: %s", cudaGetErrorString(err)); return ETPGT_ECUDA; }
    count_launch(4);
  }
  split_keys_kernel<<<grid, kThreads, 0, stream>>>(sorted, e, num_items, gcol, gptr);
  ETPGT_CHECK_LAUNCH("split_keys");
  return ETPGT_OK;
}

static size_t scan_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceScan::InclusiveSum(nullptr, bytes, (const int32_t*)nullptr, (int32_t*)nullptr, (int)n);
  return bytes;
}

extern "C" size_t etpgt_session_subgraphs_workspace_bytes(int64_t num_sessions, int64_t num_edges) {
  const int64_t b = num_sessions > 0 ? num_sessions : 1;
  const int64_t e = num_edges > 0 ? num_edges : 1;
  return 2 * align_up(b * sizeof(int32_t)) + align_up(scan_temp_bytes(b)) + 2 * align_up(e * sizeof(int32_t)) + 256;
}

static int check_sessions(const char* who, int64_t num_sessions, int max_len) {
  ETPGT_REQUIRE(num_sessions >= 0 && num_sessions < (int64_t(1) << 31), "%s: bad session count", who);
  ETPGT_REQUIRE(max_len >= 2 && max_len - 1 <= kMaxCtx, "%s: max_len must be in [2, %d]", who, kMaxCtx + 1);
  return ETPGT_OK;
}

extern "C" int etpgt_session_subgraphs_count(const int32_t* gptr, const int32_t* gcol, const int64_t* sess_ptr,
                                             const int64_t* sess_items, const int64_t* session_ids,
                                             int64_t num_sessions, int max_len,
                                             int symmetrize, int self_loop_if_empty, int32_t* node_ptr,
                                             int32_t* edge_ptr, void* ws, size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_sessions("session_subgraphs_count", num_sessions, max_len);
  if (rc != ETPGT_OK) return rc;
  if (ws_bytes < etpgt_session_subgraphs_workspace_bytes(num_sessions, 0)) {
    set_error("session_subgraphs_count: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  set_zero_kernel<<<1, 1, 0, stream>>>(node_ptr);
  set_zero_kernel<<<1, 1, 0, stream>>>(edge_ptr);
  ETPGT_CHECK_LAUNCH("set_zero");
  count_launch(1);
  if (num_sessions == 0) return ETPGT_OK;
  Workspace w(ws, ws_bytes);
  int32_t* node_cnt = w.take<int32_t>(num_sessions);
  int32_t* edge_cnt = w.take<int32_t>(num_sessions);
  size_t temp_bytes = scan_temp_bytes(num_sessions);
  void* temp = w.take<char>(temp_bytes);
  const unsigned grid = (unsigned)((num_sessions + kWarpsPerCta - 1) / kWarpsPerCta);
  session_subgraph_kernel<false><<<grid, kThreads, 0, stream>>>(gptr, gcol, nullptr, sess_ptr, sess_items, session_ids, num_sessions,
                                                               max_len, symmetrize, self_loop_if_empty, node_cnt,
                                                               edge_cnt, nullptr, nullptr, nullptr, nullptr, nullptr,
                                                               nullptr, nullptr, nullptr, nullptr);
  ETPGT_CHECK_LAUNCH("session_subgraph_count");
  cudaError_t err = cub::DeviceScan::InclusiveSum(temp, temp_bytes, node_cnt, node_ptr + 1, (int)num_sessions, stream);
  if (err == cudaSuccess)
    err = cub::DeviceScan::InclusiveSum(temp, temp_bytes, edge_cnt, edge_ptr + 1, (int)num_sessions, stream);
  if (err != cudaSuccess) { set_error("session_subgraphs scan: %s", cudaGetErrorString(err)); return ETPGT_ECUDA; }
  count_launch(4);
  return ETPGT_OK;
}

extern "C" int etpgt_session_subgraphs_fill(const int32_t* gptr, const int32_t* gcol, const int32_t* gidx,
                                            const int64_t* sess_ptr, const int64_t* sess_items,
                                            const int64_t* session_ids, int64_t num_sessions,
                                            int max_len, int symmetrize, int self_loop_if_empty,
                                            const int32_t* node_ptr, const int32_t* edge_ptr, int64_t num_edges,
                                            int64_t* x, int64_t* batch, int64_t* edge_src, int64_t* edge_dst,
                                            int64_t* target, void* ws, size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_sessions("session_subgraphs_fill", num_sessions, max_len);
  if (rc != ETPGT_OK) return rc;
  if (ws_bytes < etpgt_session_subgraphs_workspace_bytes(num_sessions, num_edges)) {
    set_error("session_subgraphs_fill: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  if (num_sessions == 0) return ETPGT_OK;
  Workspace w(ws, ws_bytes);
  int32_t* tmp_idx = w.take<int32_t>(num_edges > 0 ? num_edges : 1);
  int32_t* tmp_pair = w.take<int32_t>(num_edges > 0 ? num_edges : 1);
  const unsigned grid = (unsigned)((num_sessions + kWarpsPerCta - 1) / kWarpsPerCta);
  session_subgraph_kernel<true><<<grid, kThreads, 0, stream>>>(gptr, gcol, gidx, sess_ptr, sess_items, session_ids, num_sessions,
                                                              max_len, symmetrize, self_loop_if_empty, nullptr, nullptr,
                                                              node_ptr, edge_ptr, x, batch, edge_src, edge_dst, target,
                                                              tmp_idx, tmp_pair);
  ETPGT_CHECK_LAUNCH("session_subgraph_fill");
  return ETPGT_OK;
}

extern "C" int etpgt_sample_negatives(uint64_t seed, uint32_t step, int64_t session_base, const int64_t* sess_ptr,
                                      const int64_t* sess_items, const int64_t* session_ids,
                                      int64_t num_sessions, int max_len,
                                      int64_t num_items, int num_neg, int64_t* out, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_sessions >= 0 && num_neg >= 1 && num_items >= 2 && max_len >= 1, "sample_negatives: bad sizes");
  ETPGT_REQUIRE(num_items - 1 > max_len, "sample_negatives: catalogue must exceed the session length");
  const int64_t total = num_sessions * num_neg;
  if (total == 0) return ETPGT_OK;
  sample_negatives_kernel<<<(unsigned)((total + kThreads - 1) / kThreads), kThreads, 0, stream>>>(
      seed, step, session_base, sess_ptr, sess_items, session_ids, num_sessions, max_len, num_items, num_neg, out);
  ETPGT_CHECK_LAUNCH("sample_negatives");
  return ETPGT_OK;
}
