// In-batch negatives for the shared-pool softmax (etpgt_pool_softmax_*): the batch's targets become extra columns,
// merged with the sorted pool of etpgt_sample_item_pool, and each in-batch column gets the log-Q correction
// log(B q_i) of a streaming estimate q_i of item i's share of the batch's targets.
//
//   keys   key[b] = clamp(t_b, -1, I) + 1, val[b] = b; one stable radix sort, so equal targets keep session order
//   runs   one thread per run head of the sorted keys (n copies of item i): the estimator update
//            freq[i] = freq[i] (1 - a)^(step - last[i]) + a n / B,  last[i] = step
//          for in-range, non-padding ids only.  It equals the eager EMA q <- (1 - a) q + a f(step) applied to every
//          item every step, with the decay of the steps an item was absent applied when it next appears.
//   merge  every entry finds its output position by a binary search in the other sorted list (a merge path of one
//          element per thread).  Among equal ids the pool entries come first, then the in-batch entries in session
//          order, so identical inputs give identical bits.
//
// Out-of-range targets sort before (< 0) or after (>= I) every pool entry, never touch freq / last and get
// log_q = +inf; the padding id gets +inf too.  Those columns are never negatives.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ uint32_t column_key(int64_t id, int64_t num_items) {
  return id < 0 ? 0u : id >= num_items ? (uint32_t)(num_items + 1) : (uint32_t)(id + 1);
}

__global__ void __launch_bounds__(kThreads)
in_batch_keys_kernel(const int64_t* __restrict__ targets, int64_t batch, int64_t num_items, uint32_t* __restrict__ key,
                     int32_t* __restrict__ iota) {
  for (int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; b < batch; b += (int64_t)gridDim.x * blockDim.x) {
    key[b] = column_key(targets[b], num_items);
    iota[b] = (int32_t)b;
  }
}

// number of entries of the ascending a[0, n) that are < x (lower) or <= x (!lower)
template <typename T>
__device__ __forceinline__ int64_t rank_in(const T* __restrict__ a, int64_t n, T x, bool lower) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] < x || (!lower && a[mid] == x)) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(kThreads)
in_batch_runs_kernel(const uint32_t* __restrict__ key, int64_t batch, int64_t num_items, int64_t padding_idx,
                     int64_t step, double keep, double decay, double* __restrict__ freq, int64_t* __restrict__ last) {
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < batch; p += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t k = key[p];
    if (p > 0 && key[p - 1] == k) continue;                  // not the head of its run
    if (k == 0 || k > (uint32_t)num_items) continue;         // out of range
    const int64_t id = (int64_t)k - 1;
    if (id == padding_idx) continue;
    const int64_t n = rank_in(key + p, batch - p, k, false);
    freq[id] = freq[id] * pow(keep, (double)(step - last[id])) + decay * (double)n / (double)batch;
    last[id] = step;
  }
}

__global__ void __launch_bounds__(kThreads)
in_batch_merge_kernel(const uint32_t* __restrict__ key, const int32_t* __restrict__ sess,
                      const int64_t* __restrict__ targets, int64_t batch, const int64_t* __restrict__ pool_ids,
                      const float* __restrict__ pool_log_q, int64_t m, const double* __restrict__ freq,
                      int64_t num_items, int64_t padding_idx, int64_t* __restrict__ columns, float* __restrict__ log_q) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m + batch;
       i += (int64_t)gridDim.x * blockDim.x) {
    if (i < m) {  // pool entry: after the in-batch entries of smaller ids
      const int64_t id = pool_ids[i];
      const int64_t pos = i + rank_in(key, batch, column_key(id, num_items), true);
      columns[pos] = id;
      log_q[pos] = pool_log_q[i];
    } else {      // in-batch entry: after the pool entries of smaller or equal ids
      const int64_t j = i - m;
      const int64_t id = targets[sess[j]];
      const int64_t pos = j + rank_in(pool_ids, m, id, false);
      const bool counted = id >= 0 && id < num_items && id != padding_idx;
      columns[pos] = id;
      log_q[pos] = counted ? (float)log((double)batch * freq[id]) : INFINITY;
    }
  }
}

int key_bits(int64_t num_items) {  // the largest key is num_items + 1
  int bits = 1;
  while (bits < 32 && (int64_t(1) << bits) <= num_items + 1) ++bits;
  return bits;
}

size_t sort_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, (int)n, 0, 32);
  return bytes;
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_in_batch_columns_workspace_bytes(int64_t batch, int64_t num_pool) {
  (void)num_pool;  // the pool is read in place
  const int64_t b = batch > 0 ? batch : 1;
  return 2 * align_up(b * sizeof(uint32_t)) + 2 * align_up(b * sizeof(int32_t)) + align_up(sort_temp_bytes(b)) + 256;
}

extern "C" int etpgt_in_batch_columns(const int64_t* targets, int64_t batch, const int64_t* pool_ids,
                                      const float* pool_log_q, int64_t num_pool, double* freq, int64_t* last,
                                      int64_t num_items, int64_t padding_idx, int64_t step, double decay,
                                      int64_t* columns, float* log_q, void* ws, size_t ws_bytes,
                                      etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(batch >= 1 && batch < (int64_t(1) << 31), "in_batch_columns: batch must be in [1, 2^31) (got %lld)",
                (long long)batch);
  ETPGT_REQUIRE(num_pool >= 0 && num_pool < (int64_t(1) << 31),
                "in_batch_columns: num_pool must be in [0, 2^31) (got %lld)", (long long)num_pool);
  ETPGT_REQUIRE(num_items >= 1 && num_items < (int64_t(1) << 31),
                "in_batch_columns: num_items must be in [1, 2^31) (got %lld)", (long long)num_items);
  ETPGT_REQUIRE(padding_idx >= -1 && padding_idx < num_items, "in_batch_columns: padding_idx must be -1 or an item id");
  ETPGT_REQUIRE(decay > 0.0 && decay <= 1.0, "in_batch_columns: decay must be in (0, 1] (got %g)", decay);
  ETPGT_REQUIRE(step >= 0, "in_batch_columns: step must be >= 0 (got %lld)", (long long)step);
  ETPGT_REQUIRE(targets != nullptr && freq != nullptr && last != nullptr && columns != nullptr && log_q != nullptr,
                "in_batch_columns: targets, freq, last, columns and log_q are required");
  ETPGT_REQUIRE(num_pool == 0 || (pool_ids != nullptr && pool_log_q != nullptr),
                "in_batch_columns: pool_ids and pool_log_q are required when num_pool > 0");
  const size_t need = etpgt_in_batch_columns_workspace_bytes(batch, num_pool);
  if (ws == nullptr || ws_bytes < need) {
    set_error("in_batch_columns: workspace too small (%zu < %zu bytes)", ws_bytes, need);
    return ETPGT_EWORKSPACE;
  }
  Workspace w(ws, ws_bytes);
  uint32_t* key_in = w.take<uint32_t>(batch);
  uint32_t* key = w.take<uint32_t>(batch);
  int32_t* iota = w.take<int32_t>(batch);
  int32_t* sess = w.take<int32_t>(batch);
  size_t temp_bytes = sort_temp_bytes(batch);
  void* temp = w.take<char>(temp_bytes);
  in_batch_keys_kernel<<<grid_for(batch, kThreads, 8), kThreads, 0, stream>>>(targets, batch, num_items, key_in, iota);
  ETPGT_CHECK_LAUNCH("in_batch_keys");
  cudaError_t err = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_in, key, iota, sess, (int)batch, 0,
                                                    key_bits(num_items), stream);
  if (err != cudaSuccess) { set_error("in_batch_columns sort: %s", cudaGetErrorString(err)); return ETPGT_ECUDA; }
  count_launch(4);
  in_batch_runs_kernel<<<grid_for(batch, kThreads, 8), kThreads, 0, stream>>>(key, batch, num_items, padding_idx, step,
                                                                               1.0 - decay, decay, freq, last);
  ETPGT_CHECK_LAUNCH("in_batch_runs");
  in_batch_merge_kernel<<<grid_for(num_pool + batch, kThreads, 8), kThreads, 0, stream>>>(
      key, sess, targets, batch, pool_ids, pool_log_q, num_pool, freq, num_items, padding_idx, columns, log_q);
  ETPGT_CHECK_LAUNCH("in_batch_merge");
  return ETPGT_OK;
}
