// Deterministic "scatter-add rows by key": the backward of every item-table gather on the path
// (etpgt/model/graph_transformer.py:140 lookup; etpgt/train/losses.py:39-42 target/negative
// gathers).  torch's embedding_dense_backward sorts too; PyG-side scatter uses atomics.  Here:
// one stable radix sort of (key, position) then one owner group per distinct key adds its rows in
// ascending position order -> bit-reproducible, no atomics.
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;

__global__ void narrow_keys_iota_kernel(const int64_t* __restrict__ key64, int32_t* __restrict__ key32,
                                        int32_t* __restrict__ iota, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    key32[i] = static_cast<int32_t>(key64[i]);
    iota[i] = static_cast<int32_t>(i);
  }
}

// keys of the loss scatter: [s][0] = target of session s, [s][1 + c] = its negative c
__global__ void narrow_loss_keys_iota_kernel(const int64_t* __restrict__ targets, const int64_t* __restrict__ negatives,
                                             int64_t batch, int num_neg, int32_t* __restrict__ key32,
                                             int32_t* __restrict__ iota) {
  const int64_t n = batch * (num_neg + 1);
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = i / (num_neg + 1);
    const int c = static_cast<int>(i - s * (num_neg + 1));
    key32[i] = static_cast<int32_t>(c == 0 ? targets[s] : negatives[s * num_neg + c - 1]);
    iota[i] = static_cast<int32_t>(i);
  }
}

template <int DIM>
__global__ void __launch_bounds__(kThreads)
segment_rows_add_kernel(const int32_t* __restrict__ sorted_key, const int32_t* __restrict__ perm,
                        const float* __restrict__ coef, const float* __restrict__ src, int64_t m,
                        int src_div, int skip_key, float* __restrict__ d_table) {
  using G = RowGeom<DIM>;
  const int lane = threadIdx.x & 31;
  const int lig = lane % G::LPN;
  const int64_t groups_per_cta = (kThreads / 32) * G::GROUPS;
  const int64_t group0 = blockIdx.x * groups_per_cta + (threadIdx.x >> 5) * G::GROUPS + lane / G::LPN;
  for (int64_t p = group0; p < m; p += (int64_t)gridDim.x * groups_per_cta) {
    const int key = sorted_key[p];
    if (p > 0 && sorted_key[p - 1] == key) continue;  // not the head of its segment
    if (key == skip_key) continue;
    float4 acc[G::V];
#pragma unroll
    for (int v = 0; v < G::V; ++v) acc[v] = zero4();
    for (int64_t q = p; q < m && sorted_key[q] == key; ++q) {
      const int pos = perm[q];
      const float c = coef ? coef[pos] : 1.f;
      const float* row = src + (int64_t)(pos / src_div) * DIM;
#pragma unroll
      for (int v = 0; v < G::V; ++v) acc[v] = fma4(c, ldg4(row + 4 * (v * G::LPN + lig)), acc[v]);
    }
    float* out = d_table + (int64_t)key * DIM;
#pragma unroll
    for (int v = 0; v < G::V; ++v) {
      float* o = out + 4 * (v * G::LPN + lig);
      st4(o, add4(ld4(o), acc[v]));
    }
  }
}

int key_bits(int64_t n) {
  int bits = 1;
  while ((int64_t(1) << bits) < n && bits < 31) ++bits;
  return bits;
}

size_t sort_temp_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const int32_t*)nullptr, (int32_t*)nullptr,
                                  (const int32_t*)nullptr, (int32_t*)nullptr, static_cast<int>(n), 0, 31);
  return bytes;
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_scatter_rows_workspace_bytes(int64_t m) {
  int64_t n = m > 0 ? m : 1;
  return 4 * align_up(n * sizeof(int32_t)) + align_up(sort_temp_bytes(n)) + 256;
}

// The sort of a scatter depends on the keys only, and the keys of both scatters of a training step (the
// batch's node ids; its targets + negatives) are known as soon as the batch exists.  So the sort can be
// made ONCE per batch, next to the CSR / CSC index ("scatter plan"), off the critical path of the step.
extern "C" size_t etpgt_scatter_plan_workspace_bytes(int64_t m) {
  int64_t n = m > 0 ? m : 1;
  return 2 * align_up(n * sizeof(int32_t)) + align_up(sort_temp_bytes(n)) + 256;
}

static int scatter_plan_impl(const int64_t* keys, const int64_t* negatives, int64_t batch, int num_neg, int64_t m,
                             int64_t num_rows, int32_t* sorted_key, int32_t* perm, void* ws, size_t ws_bytes,
                             etpgt_stream_t stream_);

extern "C" int etpgt_scatter_plan(const int64_t* keys, int64_t m, int64_t num_rows, int32_t* sorted_key,
                                  int32_t* perm, void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  return scatter_plan_impl(keys, nullptr, 0, 0, m, num_rows, sorted_key, perm, ws, ws_bytes, stream);
}

extern "C" int etpgt_scatter_plan_loss(const int64_t* targets, const int64_t* negatives, int64_t batch, int num_neg,
                                       int64_t num_rows, int32_t* sorted_key, int32_t* perm, void* ws,
                                       size_t ws_bytes, etpgt_stream_t stream) {
  ETPGT_REQUIRE(batch >= 0 && num_neg >= 1 && negatives != nullptr, "scatter_plan_loss: bad arguments");
  return scatter_plan_impl(targets, negatives, batch, num_neg, batch * (num_neg + 1), num_rows, sorted_key, perm, ws,
                           ws_bytes, stream);
}

static int scatter_plan_impl(const int64_t* keys, const int64_t* negatives, int64_t batch, int num_neg, int64_t m,
                             int64_t num_rows, int32_t* sorted_key, int32_t* perm, void* ws, size_t ws_bytes,
                             etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(m >= 0 && m < (int64_t(1) << 31) && num_rows >= 1 && num_rows < (int64_t(1) << 31),
                "scatter_plan: bad size");
  if (m == 0) return ETPGT_OK;
  ETPGT_REQUIRE(keys && sorted_key && perm, "scatter_plan: null pointer");
  if (ws_bytes < etpgt_scatter_plan_workspace_bytes(m)) {
    set_error("scatter_plan: workspace %zu < %zu", ws_bytes, etpgt_scatter_plan_workspace_bytes(m));
    return ETPGT_EWORKSPACE;
  }
  Workspace w(ws, ws_bytes);
  int32_t* key_a = w.take<int32_t>(m);
  int32_t* iota = w.take<int32_t>(m);
  size_t temp_bytes = sort_temp_bytes(m);
  void* temp = w.take<char>(temp_bytes);
  if (negatives != nullptr)
    narrow_loss_keys_iota_kernel<<<grid_for(m, kThreads, 8), kThreads, 0, stream>>>(keys, negatives, batch, num_neg,
                                                                                  key_a, iota);
  else
    narrow_keys_iota_kernel<<<grid_for(m, kThreads, 8), kThreads, 0, stream>>>(keys, key_a, iota, m);
  ETPGT_CHECK_LAUNCH("scatter_plan narrow");
  cudaError_t err = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_a, sorted_key, iota, perm,
                                                    static_cast<int>(m), 0, key_bits(num_rows), stream);
  if (err != cudaSuccess) { set_error("scatter_plan sort: %s", cudaGetErrorString(err)); return ETPGT_ECUDA; }
  count_launch(4);
  return ETPGT_OK;
}

extern "C" int etpgt_scatter_rows_planned(const int32_t* sorted_key, const int32_t* perm, const float* coef,
                                          const float* src, int64_t m, int src_div, int dim, int64_t skip_key,
                                          float* d_table, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(supported_dim(dim), "scatter_rows: unsupported dim %d", dim);
  ETPGT_REQUIRE(m >= 0 && m < (int64_t(1) << 31) && src_div >= 1, "scatter_rows: bad size");
  if (m == 0) return ETPGT_OK;
  ETPGT_REQUIRE(sorted_key && perm && src && d_table, "scatter_rows_planned: null pointer");
#define CALL(D)                                                                                         \
  {                                                                                                     \
    const int64_t gpc = (kThreads / 32) * RowGeom<D>::GROUPS;                                           \
    segment_rows_add_kernel<D><<<grid_for(m, (int)gpc, 8), kThreads, 0, stream>>>(sorted_key, perm, coef, src, m, \
                                                                                 src_div, (int)skip_key, d_table); \
  }
  ETPGT_DISPATCH_DIM(dim, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("segment_rows_add");
  return ETPGT_OK;
}

extern "C" int etpgt_scatter_rows(const int64_t* keys, const float* coef, const float* src, int64_t m,
                                  int src_div, int dim, int64_t num_rows, int64_t skip_key, float* d_table,
                                  void* ws, size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  // 192 as well: the table gradient of the shared-pool softmax, whose dims are those of the tensor-core losses
  ETPGT_REQUIRE(supported_dim(dim) || dim == 192, "scatter_rows: unsupported dim %d", dim);
  ETPGT_REQUIRE(m >= 0 && m < (int64_t(1) << 31) && num_rows < (int64_t(1) << 31) && src_div >= 1,
                "scatter_rows: bad size");
  if (m == 0) return ETPGT_OK;
  if (ws_bytes < etpgt_scatter_rows_workspace_bytes(m)) {
    set_error("scatter_rows: workspace %zu < %zu", ws_bytes, etpgt_scatter_rows_workspace_bytes(m));
    return ETPGT_EWORKSPACE;
  }
  Workspace w(ws, ws_bytes);
  int32_t* key_a = w.take<int32_t>(m);
  int32_t* key_s = w.take<int32_t>(m);
  int32_t* iota = w.take<int32_t>(m);
  int32_t* perm = w.take<int32_t>(m);
  size_t temp_bytes = sort_temp_bytes(m);
  void* temp = w.take<char>(temp_bytes);
  narrow_keys_iota_kernel<<<grid_for(m, kThreads, 8), kThreads, 0, stream>>>(keys, key_a, iota, m);
  ETPGT_CHECK_LAUNCH("scatter_rows narrow");
  cudaError_t err = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, key_a, key_s, iota, perm,
                                                    static_cast<int>(m), 0, key_bits(num_rows), stream);
  if (err != cudaSuccess) { set_error("scatter_rows sort: %s", cudaGetErrorString(err)); return ETPGT_ECUDA; }
  count_launch(4);
#define CALL(D)                                                                                         \
  {                                                                                                     \
    const int64_t gpc = (kThreads / 32) * RowGeom<D>::GROUPS;                                           \
    segment_rows_add_kernel<D><<<grid_for(m, (int)gpc, 8), kThreads, 0, stream>>>(key_s, perm, coef, src, m, \
                                                                                 src_div, (int)skip_key, d_table); \
  }
  if (dim == 192) {
    CALL(192);
  } else {
    ETPGT_DISPATCH_DIM(dim, CALL)
  }
#undef CALL
  ETPGT_CHECK_LAUNCH("segment_rows_add");
  return ETPGT_OK;
}
