// a9/a10: full-catalogue scoring with a fused top-k, the exact candidate merge, and the
// Recall/NDCG accumulators.  etpgt/model/base.py:59-78 (`S @ E^T` then torch.topk),
// etpgt/utils/metrics.py:6-66.  The [B, I] score matrix is never written.
//
// This file holds the fp32 CUDA-core scorer (bit-faithful fp32 products, used for small eval
// batches and as the in-repo cross-check of the tensor-core scorer in score_tc.cu) and the
// merge / metrics kernels both scorers share.  Tie rule everywhere: higher score first, then
// LOWER item id (BASELINE.json).
#include <math.h>

#include "common.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;
constexpr int kRowsPerGroup = 4;  // register blocking: one item row is reused for 4 sessions
constexpr int kMaxK = 64;   // the fp32 scorer; the merges take k <= ETPGT_SCORE_MAX_K
constexpr int64_t kNoId = INT64_MAX;

struct Cand { float val; int32_t idx; };

// Lane groups of LPN lanes own kRowsPerGroup session rows each and scan the CTA's item chunk in
// ascending id order.  Each session keeps a sorted (desc) k-list in shared memory; a candidate
// enters only if it is strictly greater than the current k-th value, so equal scores keep the
// earlier (lower) id.
// EXCL: `excl` [batch, excl_width] lists ids each row must not receive (ascending; ids outside the
// scored range are ignored).  Every register-blocked row keeps a cursor into its list, started at the
// lower bound of the chunk's first id and advanced as the scan passes the listed ids.
template <int DIM, bool EXCL>
__global__ void __launch_bounds__(kThreads)
score_topk_f32_kernel(const float* __restrict__ sess, const float* __restrict__ table, int64_t batch,
                      int64_t num_items, int k, int64_t chunk, int64_t id_base, int parts,
                      float* __restrict__ cand_val, int64_t* __restrict__ cand_idx,
                      const int64_t* __restrict__ excl, int64_t excl_width) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  constexpr int GROUPS_PER_CTA = (kThreads / 32) * G::GROUPS;
  extern __shared__ Cand lists[];  // [GROUPS_PER_CTA * kRowsPerGroup][k]
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int group = (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
  const unsigned gmask = LPN == 32 ? 0xffffffffu : (((1u << (LPN % 32)) - 1u) << ((lane / LPN) * LPN));
  const int64_t row0 =((int64_t)blockIdx.y * GROUPS_PER_CTA + group) * kRowsPerGroup;
  const int64_t begin = blockIdx.x * chunk;
  const int64_t end = begin + chunk < num_items ? begin + chunk : num_items;

  float4 s[kRowsPerGroup][V];
  float thr[kRowsPerGroup];
  Cand* mine[kRowsPerGroup];
#pragma unroll
  for (int r = 0; r < kRowsPerGroup; ++r) {
    const int64_t row = row0 + r < batch ? row0 + r : batch - 1;
#pragma unroll
    for (int v = 0; v < V; ++v) s[r][v] = ldg4(sess + row * DIM + 4 * (v * LPN + lig));
    mine[r] = lists + ((size_t)group * kRowsPerGroup + r) * k;
    for (int t = lig; t < k; t += LPN) mine[r][t] = Cand{-INFINITY, -1};
    thr[r] = -INFINITY;
  }
  __syncwarp();
  int filled[kRowsPerGroup] = {0, 0, 0, 0};
  const int64_t* ex_next[kRowsPerGroup];   // EXCL: the row's next listed id >= the scan position
  const int64_t* ex_end[kRowsPerGroup];
  if (EXCL) {
#pragma unroll
    for (int r = 0; r < kRowsPerGroup; ++r) {
      const int64_t row = row0 + r < batch ? row0 + r : batch - 1;
      const int64_t* ids = excl + row * excl_width;
      int64_t lo = 0, hi = excl_width;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (ids[mid] < id_base + begin) lo = mid + 1;
        else hi = mid;
      }
      ex_next[r] = ids + lo;
      ex_end[r] = ids + excl_width;
    }
  }

  for (int64_t item = begin; item < end; ++item) {
    float4 e[V];
#pragma unroll
    for (int v = 0; v < V; ++v) e[v] = ldg4(table + item * DIM + 4 * (v * LPN + lig));
#pragma unroll
    for (int r = 0; r < kRowsPerGroup; ++r) {
      float part = 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) part += dot4(s[r][v], e[v]);
      const float sc = group_sum<LPN>(part);
      bool listed = false;   // uniform within the lane group (one row, one item)
      if (EXCL) {
        while (ex_next[r] < ex_end[r] && *ex_next[r] <= id_base + item) {
          listed = listed || *ex_next[r] == id_base + item;
          ++ex_next[r];
        }
      }
      // enters while the list is not full, or when strictly better than the k-th entry
      if (!listed && (filled[r] < k || sc > thr[r])) {
        if (lig == 0) {
          int t = filled[r] < k ? filled[r] : k - 1;
          while (t > 0 && mine[r][t - 1].val < sc) { mine[r][t] = mine[r][t - 1]; --t; }
          mine[r][t] = Cand{sc, (int32_t)(item - begin)};
        }
        if (filled[r] < k) ++filled[r];
        __syncwarp(gmask);  // the branch is uniform within a lane group, not within the warp
        thr[r] = filled[r] < k ? -INFINITY : mine[r][k - 1].val;
      }
    }
  }
  __syncwarp();
#pragma unroll
  for (int r = 0; r < kRowsPerGroup; ++r) {
    const int64_t row = row0 + r;
    if (row >= batch) continue;
    for (int t = lig; t < k; t += LPN) {
      const Cand c = mine[r][t];
      const int64_t o = (row * parts + blockIdx.x) * k + t;
      cand_val[o] = c.idx < 0 ? -INFINITY : c.val;
      cand_idx[o] = c.idx < 0 ? kNoId : id_base + begin + c.idx;
    }
  }
}

__device__ __forceinline__ bool better(float v, int64_t i, float bv, int64_t bi) {
  return v > bv || (v == bv && i < bi);
}

// One warp per row: k selection passes over the row's candidates; pass t takes the best
// candidate that comes strictly after the previous winner in (score desc, id asc) order.
__global__ void __launch_bounds__(kThreads)
topk_merge_kernel(const float* __restrict__ cand_val, const int64_t* __restrict__ cand_idx, int64_t batch,
                  int64_t m, int k, float* __restrict__ top_val, int64_t* __restrict__ top_idx) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5;
  if (row >= batch) return;
  const float* cv = cand_val + row * m;
  const int64_t* ci = cand_idx + row * m;
  float prev_v = INFINITY;
  int64_t prev_i = -1;
  for (int t = 0; t < k; ++t) {
    float bv = -INFINITY;
    int64_t bi = kNoId;
    for (int64_t c = lane; c < m; c += 32) {
      const float v = cv[c];
      const int64_t i = ci[c];
      const bool after_prev = v < prev_v || (v == prev_v && i > prev_i);
      if (after_prev && better(v, i, bv, bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { top_val[row * k + t] = bv; top_idx[row * k + t] = bi; }
    prev_v = bv;
    prev_i = bi;
  }
}

__global__ void __launch_bounds__(1024)
topk_metrics_kernel(const int64_t* __restrict__ top_idx, const int64_t* __restrict__ targets, int64_t batch,
                    int k_stride, int k, double* __restrict__ out) {
  __shared__ double red[2][1024];
  double hits = 0, gain = 0;
  for (int64_t b = threadIdx.x; b < batch; b += 1024) {
    const int64_t t = targets[b];
    for (int p = 0; p < k; ++p) {
      if (top_idx[b * k_stride + p] == t) {  // first match: metrics.py:49 argmax
        hits += 1.0;
        gain += 1.0 / log2((double)p + 2.0);
        break;
      }
    }
  }
  red[0][threadIdx.x] = hits;
  red[1][threadIdx.x] = gain;
  __syncthreads();
  for (int off = 512; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) {
      red[0][threadIdx.x] += red[0][threadIdx.x + off];
      red[1][threadIdx.x] += red[1][threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { out[0] += red[0][0]; out[1] += red[1][0]; }
}

// Item-sharded evaluation: the candidates of shard p for ALL sessions arrive as one packed block
// (val [rows_total, k] f32 | idx [rows_total, k] i64) per rank, gathered rank-major by ONE collective; this merges
// the rows [row_begin, row_begin + rows) straight out of that layout (no transposes / concatenations in between)
// and, when targets are given, notes where each target sits in the merged list (-1: not in the top-k).
__global__ void __launch_bounds__(kThreads)
topk_merge_parts_kernel(const char* __restrict__ parts, int num_parts, size_t part_stride, size_t idx_offset, int k,
                        int64_t row_begin, int64_t rows, float* __restrict__ top_val, int64_t* __restrict__ top_idx,
                        const int64_t* __restrict__ targets, int32_t* __restrict__ hit_pos) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5;
  if (row >= rows) return;
  const int64_t src = (row_begin + row) * k;
  const int m = num_parts * k;
  const int64_t target = targets != nullptr ? targets[row] : kNoId;
  int found = -1;
  float prev_v = INFINITY;
  int64_t prev_i = -1;
  for (int t = 0; t < k; ++t) {
    float bv = -INFINITY;
    int64_t bi = kNoId;
    for (int c = lane; c < m; c += 32) {
      const char* part = parts + (size_t)(c / k) * part_stride;
      const float v = reinterpret_cast<const float*>(part)[src + c % k];
      const int64_t i = reinterpret_cast<const int64_t*>(part + idx_offset)[src + c % k];
      const bool after_prev = v < prev_v || (v == prev_v && i > prev_i);
      if (after_prev && better(v, i, bv, bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { top_val[row * k + t] = bv; top_idx[row * k + t] = bi; }
    if (found < 0 && bi == target) found = t;   // first match: metrics.py:49 argmax
    prev_v = bv;
    prev_i = bi;
  }
  if (lane == 0 && hit_pos != nullptr) hit_pos[row] = found;
}

// k > 64: one CTA per row.  Candidates that beat the bar are appended to a shared buffer of kWideBuf (score, id)
// pairs; whenever the next block of 256 could overflow it, the buffer is bitonic-sorted by (score desc, id asc), exact
// duplicates are dropped (as the selection passes above drop them) and it is cut to the best k, whose last pair
// becomes the bar.  A row costs a few sorts instead of k passes over its parts * k candidates.
constexpr int kWideBuf = 2048;

__device__ void wide_sort_pairs(float* sv, int64_t* si, int n) {
  int p = 1;
  while (p < n) p <<= 1;
  for (int i = n + (int)threadIdx.x; i < p; i += kThreads) { sv[i] = -INFINITY; si[i] = kNoId; }
  __syncthreads();
  for (int size = 2; size <= p; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = threadIdx.x; t < p / 2; t += kThreads) {
        const int lo = (t / stride) * 2 * stride + (t % stride), hi = lo + stride;
        const bool desc = (lo & size) == 0;
        const float av = sv[lo], bv = sv[hi];
        const int64_t ai = si[lo], bi = si[hi];
        if (better(bv, bi, av, ai) == desc) { sv[lo] = bv; si[lo] = bi; sv[hi] = av; si[hi] = ai; }
      }
      __syncthreads();
    }
  }
}

// Whole CTA: sorts, de-duplicates and cuts the buffer to k once it could overflow (force: always); returns the
// number of pairs kept and sets the bar once k are known.
__device__ int wide_cut(float* sv, int64_t* si, int* s_n, int k, bool force, bool& have_bar, float& bar_v,
                        int64_t& bar_i) {
  __syncthreads();
  int n = *s_n;
  __syncthreads();
  if (!force && n <= kWideBuf - kThreads) return n;
  wide_sort_pairs(sv, si, n);
  if (threadIdx.x < 32) {   // compaction by warp 0: writes never pass the chunk being read
    const int lane = threadIdx.x;
    int kept = 0;
    float cv = 0.f;
    int64_t ci = 0;
    for (int c0 = 0; c0 < n && kept < k; c0 += 32) {
      const int c = c0 + lane;
      const float v = c < n ? sv[c] : 0.f;
      const int64_t i = c < n ? si[c] : 0;
      float pv = __shfl_up_sync(0xffffffffu, v, 1);
      int64_t pi = __shfl_up_sync(0xffffffffu, i, 1);
      if (lane == 0) { pv = cv; pi = ci; }
      const bool keep = c < n && (c == 0 || !(pv == v && pi == i));
      cv = __shfl_sync(0xffffffffu, v, 31);
      ci = __shfl_sync(0xffffffffu, i, 31);
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      const int pos = kept + __popc(m & ((1u << lane) - 1));
      __syncwarp();
      if (keep && pos < k) { sv[pos] = v; si[pos] = i; }
      kept += __popc(m);
      __syncwarp();
    }
    if (lane == 0) *s_n = kept < k ? kept : k;
  }
  __syncthreads();
  n = *s_n;
  if (n == k) { have_bar = true; bar_v = sv[k - 1]; bar_i = si[k - 1]; }
  __syncthreads();
  return n;
}

// PARTS: the rank-major layout of topk_merge_parts_kernel; otherwise [batch, m] candidate arrays.
template <bool PARTS>
__global__ void __launch_bounds__(kThreads)
topk_merge_wide_kernel(const float* __restrict__ cand_val, const int64_t* __restrict__ cand_idx, int64_t m,
                       const char* __restrict__ parts, int num_parts, size_t part_stride, size_t idx_offset,
                       int64_t row_begin, int k, float* __restrict__ top_val, int64_t* __restrict__ top_idx,
                       const int64_t* __restrict__ targets, int32_t* __restrict__ hit_pos) {
  __shared__ float sv[kWideBuf];
  __shared__ int64_t si[kWideBuf];
  __shared__ int s_n, s_found;
  const int64_t row = blockIdx.x;
  const int64_t total = PARTS ? (int64_t)num_parts * k : m;
  const int64_t src = (row_begin + row) * k;
  if (threadIdx.x == 0) { s_n = 0; s_found = INT_MAX; }
  __syncthreads();
  bool have_bar = false;
  float bar_v = -INFINITY;
  int64_t bar_i = kNoId;
  for (int64_t c0 = 0; c0 < total; c0 += kThreads) {
    const int64_t c = c0 + threadIdx.x;
    if (c < total) {
      float v;
      int64_t i;
      if (PARTS) {
        const char* part = parts + (size_t)(c / k) * part_stride;
        v = reinterpret_cast<const float*>(part)[src + c % k];
        i = reinterpret_cast<const int64_t*>(part + idx_offset)[src + c % k];
      } else {
        v = cand_val[row * m + c];
        i = cand_idx[row * m + c];
      }
      if (!have_bar || better(v, i, bar_v, bar_i)) {
        const int pos = atomicAdd(&s_n, 1);
        sv[pos] = v;
        si[pos] = i;
      }
    }
    wide_cut(sv, si, &s_n, k, false, have_bar, bar_v, bar_i);
  }
  const int n = wide_cut(sv, si, &s_n, k, true, have_bar, bar_v, bar_i);
  const int64_t target = targets != nullptr ? targets[row] : kNoId;
  for (int t = threadIdx.x; t < k; t += kThreads) {
    const float v = t < n ? sv[t] : -INFINITY;
    const int64_t i = t < n ? si[t] : kNoId;
    top_val[row * k + t] = v;
    top_idx[row * k + t] = i;
    if (targets != nullptr && i == target) atomicMin(&s_found, t);
  }
  __syncthreads();
  if (threadIdx.x == 0 && hit_pos != nullptr) hit_pos[row] = s_found == INT_MAX ? -1 : s_found;
}

// hit_pos[b] = position of the target in the top-k (-1: missed) -> acc[0] += #hits within k, acc[1] += sum of
// 1/log2(pos + 2) over them (etpgt/utils/metrics.py:6-66); one CTA, fixed order: deterministic.
__global__ void __launch_bounds__(1024)
hit_metrics_kernel(const int32_t* __restrict__ hit_pos, int64_t batch, int k, double* __restrict__ out) {
  __shared__ double red[2][1024];
  double hits = 0, gain = 0;
  for (int64_t b = threadIdx.x; b < batch; b += 1024) {
    const int p = hit_pos[b];
    if (p >= 0 && p < k) {
      hits += 1.0;
      gain += 1.0 / log2((double)p + 2.0);
    }
  }
  red[0][threadIdx.x] = hits;
  red[1][threadIdx.x] = gain;
  __syncthreads();
  for (int off = 512; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) {
      red[0][threadIdx.x] += red[0][threadIdx.x + off];
      red[1][threadIdx.x] += red[1][threadIdx.x + off];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { out[0] += red[0][0]; out[1] += red[1][0]; }
}

struct ScorePlan {
  int parts;
  int64_t chunk;
  int row_blocks;
};

template <int DIM>
ScorePlan plan_for(int64_t batch, int64_t num_items, int k) {
  constexpr int rows_per_cta = (kThreads / 32) * RowGeom<DIM>::GROUPS * kRowsPerGroup;
  ScorePlan p;
  p.row_blocks = (int)((batch + rows_per_cta - 1) / rows_per_cta);
  int64_t want = (2 * kNumSMs + p.row_blocks - 1) / p.row_blocks;  // about two waves of CTAs
  int64_t min_chunk = 4 * (int64_t)k > 256 ? 4 * (int64_t)k : 256;
  int64_t max_parts = (num_items + min_chunk - 1) / min_chunk;
  if (want > max_parts) want = max_parts;
  if (want < 1) want = 1;
  p.chunk = (num_items + want - 1) / want;
  p.parts = (int)((num_items + p.chunk - 1) / p.chunk);
  return p;
}

ScorePlan plan_dispatch(int64_t batch, int64_t num_items, int dim, int k) {
  switch (dim) {
    case 32: return plan_for<32>(batch, num_items, k);
    case 64: return plan_for<64>(batch, num_items, k);
    case 128: return plan_for<128>(batch, num_items, k);
    default: return plan_for<256>(batch, num_items, k);
  }
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_score_topk_workspace_bytes(int64_t batch, int64_t num_items, int dim, int k) {
  if (batch <= 0 || num_items <= 0 || k <= 0) return 256;
  const ScorePlan p = plan_dispatch(batch, num_items, dim, k);
  const size_t m = (size_t)batch * p.parts * k;
  return align_up(m * sizeof(float)) + align_up(m * sizeof(int64_t)) + 256;
}

extern "C" int etpgt_topk_merge(const float* cand_val, const int64_t* cand_idx, int64_t batch, int parts, int k,
                                float* top_val, int64_t* top_idx, etpgt_stream_t stream) {
  ETPGT_REQUIRE(batch >= 0 && parts >= 1 && k >= 1 && k <= ETPGT_SCORE_MAX_K, "topk_merge: bad sizes (k <= %d)",
                ETPGT_SCORE_MAX_K);
  if (batch == 0) return ETPGT_OK;
  if (k > kMaxK) {
    topk_merge_wide_kernel<false><<<(unsigned)batch, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        cand_val, cand_idx, (int64_t)parts * k, nullptr, 0, 0, 0, 0, k, top_val, top_idx, nullptr, nullptr);
    ETPGT_CHECK_LAUNCH("topk_merge_wide");
    return ETPGT_OK;
  }
  const int64_t warps_per_cta = kThreads / 32;
  topk_merge_kernel<<<(unsigned)((batch + warps_per_cta - 1) / warps_per_cta), kThreads, 0,
                      static_cast<cudaStream_t>(stream)>>>(cand_val, cand_idx, batch, (int64_t)parts * k, k, top_val,
                                                           top_idx);
  ETPGT_CHECK_LAUNCH("topk_merge");
  return ETPGT_OK;
}

namespace {

// The scorer behind etpgt_score_topk_f32 (excl == nullptr) and etpgt_score_topk_f32_exclude (k_any: k may exceed the
// eligible items, whose missing slots become (-inf, INT64_MAX) sentinels).
int score_topk_f32_run(const float* sess, const float* table, int64_t batch, int64_t num_items, int dim, int k,
                       int64_t id_base, float* top_val, int64_t* top_idx, const int64_t* excl, int64_t excl_width,
                       bool k_any, void* ws, size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(supported_dim(dim), "score_topk: unsupported dim %d", dim);
  ETPGT_REQUIRE(batch >= 0 && num_items >= 1, "score_topk: bad sizes");
  if (k_any) {
    ETPGT_REQUIRE(k >= 1 && k <= kMaxK,
                  "score_topk: k=%d must be in [1, %d] for the fp32 scorer (the bf16 scorer takes k <= %d)", k, kMaxK,
                  ETPGT_SCORE_MAX_K);
  } else {
    ETPGT_REQUIRE(k >= 1 && k <= kMaxK && k <= num_items,
                  "score_topk: k=%d must be in [1, min(%d, num_items)] for the fp32 scorer (the bf16 scorer takes k <= "
                  "%d)", k, kMaxK, ETPGT_SCORE_MAX_K);
  }
  if (ws_bytes < etpgt_score_topk_workspace_bytes(batch, num_items, dim, k)) {
    set_error("score_topk: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  if (batch == 0) return ETPGT_OK;
  const ScorePlan p = plan_dispatch(batch, num_items, dim, k);
  Workspace w(ws, ws_bytes);
  const size_t m = (size_t)batch * p.parts * k;
  float* cand_val = w.take<float>(m);
  int64_t* cand_idx = w.take<int64_t>(m);
#define CALL2(D, EX)                                                                                         \
  {                                                                                                          \
    const size_t smem = (size_t)(kThreads / 32) * RowGeom<D>::GROUPS * kRowsPerGroup * k * sizeof(Cand);     \
    if (smem > 48 * 1024)                                                                                    \
      cudaFuncSetAttribute(score_topk_f32_kernel<D, EX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    score_topk_f32_kernel<D, EX><<<dim3(p.parts, p.row_blocks), kThreads, smem, stream>>>(                    \
        sess, table, batch, num_items, k, p.chunk, id_base, p.parts, cand_val, cand_idx, excl, excl_width);  \
  }
#define CALL(D)                             \
  {                                         \
    if (excl != nullptr) CALL2(D, true)     \
    else CALL2(D, false)                    \
  }
  ETPGT_DISPATCH_DIM(dim, CALL)
#undef CALL
#undef CALL2
  ETPGT_CHECK_LAUNCH("score_topk_f32");
  return etpgt_topk_merge(cand_val, cand_idx, batch, p.parts, k, top_val, top_idx, stream_);
}

}  // namespace

extern "C" int etpgt_score_topk_f32(const float* sess, const float* table, int64_t batch, int64_t num_items, int dim,
                                    int k, int64_t id_base, float* top_val, int64_t* top_idx, void* ws,
                                    size_t ws_bytes, etpgt_stream_t stream) {
  return score_topk_f32_run(sess, table, batch, num_items, dim, k, id_base, top_val, top_idx, nullptr, 0, false, ws,
                            ws_bytes, stream);
}

extern "C" int etpgt_score_topk_f32_exclude(const float* sess, const float* table, int64_t batch, int64_t num_items,
                                            int dim, int k, int64_t id_base, float* top_val, int64_t* top_idx,
                                            const int64_t* exclude, int64_t exclude_width, void* ws, size_t ws_bytes,
                                            etpgt_stream_t stream) {
  ETPGT_REQUIRE(exclude_width >= 0, "score_topk_exclude: negative exclude_width");
  ETPGT_REQUIRE(exclude_width == 0 || batch == 0 || exclude != nullptr, "score_topk_exclude: null exclude list");
  return score_topk_f32_run(sess, table, batch, num_items, dim, k, id_base, top_val, top_idx,
                            exclude_width > 0 ? exclude : nullptr, exclude_width, true, ws, ws_bytes, stream);
}

extern "C" int etpgt_topk_metrics(const int64_t* top_idx, const int64_t* targets, int64_t batch, int k_stride, int k,
                                  double* out, etpgt_stream_t stream) {
  ETPGT_REQUIRE(batch >= 0 && k >= 1 && k <= k_stride, "topk_metrics: bad sizes");
  topk_metrics_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(top_idx, targets, batch, k_stride, k, out);
  ETPGT_CHECK_LAUNCH("topk_metrics");
  return ETPGT_OK;
}

extern "C" int etpgt_topk_merge_parts(const void* parts, int num_parts, size_t part_stride, size_t idx_offset,
                                      int64_t rows_total, int k, int64_t row_begin, int64_t rows, float* top_val,
                                      int64_t* top_idx, const int64_t* targets, int32_t* hit_pos,
                                      etpgt_stream_t stream) {
  ETPGT_REQUIRE(num_parts >= 1 && num_parts <= 64 && k >= 1 && k <= ETPGT_SCORE_MAX_K,
                "topk_merge_parts: bad sizes (k <= %d)", ETPGT_SCORE_MAX_K);
  ETPGT_REQUIRE(rows >= 0 && row_begin >= 0 && row_begin + rows <= rows_total, "topk_merge_parts: bad row range");
  ETPGT_REQUIRE(idx_offset % 8 == 0 && part_stride % 8 == 0 && idx_offset >= (size_t)rows_total * k * sizeof(float) &&
                    part_stride >= idx_offset + (size_t)rows_total * k * sizeof(int64_t),
                "topk_merge_parts: bad part layout");
  ETPGT_REQUIRE(rows == 0 || (parts && top_val && top_idx), "topk_merge_parts: null pointer");
  ETPGT_REQUIRE((targets == nullptr) == (hit_pos == nullptr), "topk_merge_parts: targets and hit_pos come together");
  if (rows == 0) return ETPGT_OK;
  if (k > kMaxK) {
    topk_merge_wide_kernel<true><<<(unsigned)rows, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        nullptr, nullptr, 0, static_cast<const char*>(parts), num_parts, part_stride, idx_offset, row_begin, k, top_val,
        top_idx, targets, hit_pos);
    ETPGT_CHECK_LAUNCH("topk_merge_parts_wide");
    return ETPGT_OK;
  }
  const int64_t warps_per_cta = kThreads / 32;
  topk_merge_parts_kernel<<<(unsigned)((rows + warps_per_cta - 1) / warps_per_cta), kThreads, 0,
                            static_cast<cudaStream_t>(stream)>>>(static_cast<const char*>(parts), num_parts,
                                                                 part_stride, idx_offset, k, row_begin, rows, top_val,
                                                                 top_idx, targets, hit_pos);
  ETPGT_CHECK_LAUNCH("topk_merge_parts");
  return ETPGT_OK;
}

extern "C" int etpgt_hit_metrics(const int32_t* hit_pos, int64_t batch, int k, double* out, etpgt_stream_t stream) {
  ETPGT_REQUIRE(batch >= 0 && k >= 1 && out && (batch == 0 || hit_pos), "hit_metrics: bad arguments");
  hit_metrics_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(hit_pos, batch, k, out);
  ETPGT_CHECK_LAUNCH("hit_metrics");
  return ETPGT_OK;
}
