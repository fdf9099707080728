// a5, hub rows: the fused TransformerConv passes for destinations / sources with more than kHubThreshold edges.
//
// The row kernels of tconv.cu give one lane group a whole row and walk its edges serially — right for session
// batches (rows of a few edges) and for the bulk of a co-occurrence graph, hopeless for the head of a power-law
// degree distribution: the reference's synthetic generator draws items zipf(1.5)
// (scripts/data/00_generate_synthetic_data.py:53), the RetailRocket-shaped graph has rows of several hundred edges
// and the 1M-item graph rows of 80,000.  Here such a row is cut into chunks of kHubChunk edges (etpgt_hub_plan:
// prefix sums over the row pointers, deterministic).  ONE CTA takes a chunk: the row's query (backward: query and
// d_agg) is staged once in shared memory, each of the CTA's lane groups walks a slice of the chunk with exactly the
// per-edge arithmetic of the row kernels (tconv.cuh), and the groups' partials — forward (m, l, acc) with the
// softmax rescaling, backward plain sums — are combined in group order through shared memory into one partial per
// chunk.  A second kernel combines the chunks of a row in chunk order and finishes the row (forward: normalise,
// gate, outputs; backward: gradient rows, column sums).  No atomics anywhere: results are bit-reproducible.
//
// HBM-bound like the row kernels: the partials add (dim + 16) * 4 B per 256 edges (0.2 % of the gathered bytes).
#include <cub/device/device_scan.cuh>

#include "tconv.cuh"

namespace etpgt {
namespace {

constexpr int kPartPad = 16;   // forward partial row: acc [DIM] | m [8] | l [8]

template <int DIM>
struct HubGeom {
  using G = RowGeom<DIM>;
  static constexpr int NG = (kThreads / 32) * G::GROUPS;   // lane groups per CTA
  static constexpr int PER = kHubChunk / NG;               // edges of a chunk per lane group
  static_assert(kHubChunk % NG == 0 && PER >= 1, "chunk must split evenly over the lane groups");
};

// ------------------------------------------------------------------------------- plan
// val[n] = (1 << 32 | chunks) for a hub row, else 0: ONE exclusive prefix sum numbers hub rows (high word) and
// their chunks (low word) at once.
__global__ void hub_flags_kernel(const int32_t* __restrict__ ptr, int64_t num_nodes, unsigned long long* __restrict__ val) {
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    const int deg = ptr[n + 1] - ptr[n];
    val[n] = deg > kHubThreshold ? ((1ull << 32) | (unsigned long long)((deg + kHubChunk - 1) / kHubChunk)) : 0ull;
  }
}

__global__ void hub_emit_kernel(const int32_t* __restrict__ ptr, int64_t num_nodes,
                                const unsigned long long* __restrict__ val, const unsigned long long* __restrict__ offset,
                                HubRow* __restrict__ rows, HubChunk* __restrict__ chunks, int32_t* __restrict__ counts) {
  for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < num_nodes; n += (int64_t)gridDim.x * blockDim.x) {
    const unsigned long long v = val[n], o = offset[n];
    if (n == num_nodes - 1) {
      counts[0] = (int32_t)((o + v) >> 32);
      counts[1] = (int32_t)((o + v) & 0xffffffffull);
    }
    if (v == 0) continue;
    const int slot = (int)(o >> 32), first = (int)(o & 0xffffffffull), nch = (int)(v & 0xffffffffull);
    const int begin = ptr[n], deg = ptr[n + 1] - begin;
    rows[slot] = HubRow{(int32_t)n, first, nch, 0};
    for (int c = 0; c < nch; ++c) {
      const int b = c * kHubChunk;
      chunks[first + c] = HubChunk{(int32_t)n, begin + b, min(kHubChunk, deg - b), slot};
    }
  }
}

// ------------------------------------------------------------------------------- forward
template <int DIM, int HEAD_DIM>
__global__ void __launch_bounds__(kThreads, 2)
tconv_fwd_hub_chunk_kernel(const float* __restrict__ qkvs, const int32_t* __restrict__ col,
                           const int32_t* __restrict__ eperm, const float* __restrict__ alpha_mask,
                           const int32_t* __restrict__ num_chunks_ptr, const HubChunk* __restrict__ chunks,
                           float* __restrict__ partial /* [chunks][DIM + kPartPad] */) {
  using G = RowGeom<DIM>;
  using H = HubGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN, NG = H::NG, PER = H::PER;
  constexpr int HEAD_F4 = HEAD_DIM / 4;
  constexpr int STRIDE = DIM + kPartPad;
  __shared__ __align__(16) float q_s[DIM];
  __shared__ __align__(16) float part_s[NG * STRIDE];
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int group = (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
  const int num_chunks = *num_chunks_ptr;
  for (int c = blockIdx.x; c < num_chunks; c += gridDim.x) {
    const HubChunk ch = chunks[c];
    // the hub's query row, staged once for all lane groups of the CTA
    for (int i = threadIdx.x; i < DIM / 4; i += kThreads) st4(q_s + 4 * i, ldg4(qkvs + (int64_t)ch.node * 4 * DIM + 4 * i));
    __syncthreads();
    float4 q[V];
#pragma unroll
    for (int v = 0; v < V; ++v) q[v] = ld4(q_s + 4 * (v * LPN + lig));
    const int b = min(group * PER, ch.edge_count);
    const int cnt = min(PER, ch.edge_count - b);
    int cnt_max = cnt;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt_max = max(cnt_max, __shfl_xor_sync(0xffffffffu, cnt_max, off));
    float m[V], l[V];
    float4 acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { m[v] = -INFINITY; l[v] = 0.f; acc[v] = zero4(); }
    const EdgeMeta meta = load_edge_meta(col, alpha_mask != nullptr ? eperm : nullptr, ch.edge_begin + b, cnt, 0, lig);
    fwd_edges<DIM, HEAD_DIM, kEdgeUnroll>(qkvs, q, col, eperm, alpha_mask, ch.edge_begin + b, cnt, cnt_max, ch.node, lig,
                                          meta, m, l, acc);
    float* mine = part_s + group * STRIDE;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int f = v * LPN + lig;
      st4(mine + 4 * f, acc[v]);
      if (f % HEAD_F4 == 0) { mine[DIM + f / HEAD_F4] = m[v]; mine[DIM + 8 + f / HEAD_F4] = l[v]; }
    }
    __syncthreads();
    // (m, l, acc) of the lane groups combined in group order; thread t owns float4 column t
    if (threadIdx.x < DIM / 4) {
      const int f = threadIdx.x, h = f / HEAD_F4;
      float big = -INFINITY;
      for (int g = 0; g < NG; ++g) big = fmaxf(big, part_s[g * STRIDE + DIM + h]);
      float lsum = 0.f;
      float4 a = zero4();
      for (int g = 0; g < NG; ++g) {
        const float w = expf(part_s[g * STRIDE + DIM + h] - big);   // a group without edges has m = -inf: weight 0
        lsum += part_s[g * STRIDE + DIM + 8 + h] * w;
        a = fma4(w, ld4(part_s + g * STRIDE + 4 * f), a);
      }
      float* dst = partial + (int64_t)c * STRIDE;
      st4(dst + 4 * f, a);
      if (f % HEAD_F4 == 0) { dst[DIM + h] = big; dst[DIM + 8 + h] = lsum; }
    }
    __syncthreads();   // shared memory is reused by the next chunk
  }
}

template <int DIM, int HEAD_DIM>
__global__ void __launch_bounds__(kThreads)
tconv_fwd_hub_combine_kernel(const float* __restrict__ qkvs, const int32_t* __restrict__ num_rows_ptr,
                             const HubRow* __restrict__ rows, const float* __restrict__ partial,
                             const float* __restrict__ w_beta, float* __restrict__ out, float* __restrict__ agg_out,
                             float* __restrict__ beta_out, float* __restrict__ m_out, float* __restrict__ invl_out,
                             double* __restrict__ stat_rows /* [gridDim.x][2*DIM] or NULL */) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN, NG = HubGeom<DIM>::NG;
  constexpr int STRIDE = DIM + kPartPad;
  extern __shared__ double stat_s[];   // [NG][2*DIM] when stat_rows != NULL
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int num_rows = *num_rows_ptr;
  double* stat_mine = nullptr;
  if (stat_rows != nullptr) {
    stat_mine = stat_s + (size_t)((threadIdx.x >> 5) * G::GROUPS + lane / LPN) * 2 * DIM;
#pragma unroll
    for (int v = 0; v < V; ++v)
#pragma unroll
      for (int c = 0; c < 4; ++c) { stat_mine[4 * (v * LPN + lig) + c] = 0.0; stat_mine[DIM + 4 * (v * LPN + lig) + c] = 0.0; }
  }
  for (int base = blockIdx.x * NG; base < num_rows; base += gridDim.x * NG) {
    const int warp_base = base + (threadIdx.x >> 5) * G::GROUPS;
    if (warp_base >= num_rows) continue;   // warp-uniform
    const int slot = warp_base + lane / LPN;
    const bool valid = slot < num_rows;
    const HubRow r = valid ? rows[slot] : HubRow{0, 0, 0, 0};
    float m[V], l[V];
    float4 acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { m[v] = -INFINITY; l[v] = 0.f; acc[v] = zero4(); }
    constexpr int kAhead = 4;   // chunk partials loaded ahead of the (ordered) merge: a long row is a chain of loads
    for (int c0 = 0; c0 < r.num_chunks; c0 += kAhead) {
      float mc[kAhead][V], lc[kAhead][V];
      float4 a[kAhead][V];
#pragma unroll
      for (int u = 0; u < kAhead; ++u) {
        const int c = min(c0 + u, r.num_chunks - 1);
        const float* src = partial + (int64_t)(r.first_chunk + c) * STRIDE;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const int h = head_of<DIM, HEAD_DIM>(v, lig);
          mc[u][v] = src[DIM + h];
          lc[u][v] = src[DIM + 8 + h];
          a[u][v] = ldg4(src + 4 * (v * LPN + lig));
        }
      }
#pragma unroll
      for (int u = 0; u < kAhead; ++u) {   // chunk order: deterministic
        if (c0 + u >= r.num_chunks) break;
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float m_new = fmaxf(m[v], mc[u][v]);
          const float w0 = expf(m[v] - m_new), w1 = expf(mc[u][v] - m_new);
          l[v] = l[v] * w0 + lc[u][v] * w1;
          acc[v] = fma4(w1, a[u][v], scale4(w0, acc[v]));
          m[v] = m_new;
        }
      }
    }
    const int64_t nrow = r.node;
    float4 xr[V];
    load_row<DIM>(qkvs + nrow * 4 * DIM + 3 * DIM, lig, xr);
    fwd_epilogue<DIM, HEAD_DIM>(xr, valid, nrow, lig, m, l, acc, w_beta, out, agg_out, beta_out, m_out,
                                invl_out, stat_mine);
  }
  if (stat_rows != nullptr) stats_flush<DIM>(stat_s, stat_rows + (size_t)blockIdx.x * 2 * DIM);
}

// ------------------------------------------------------------------------------- backward, destination side
template <int DIM, int HEAD_DIM>
__global__ void __launch_bounds__(kThreads, 2)
tconv_bwd_dst_hub_chunk_kernel(const float* __restrict__ qkvs, const int32_t* __restrict__ col,
                               const int32_t* __restrict__ eperm, const float* __restrict__ alpha_mask,
                               const float* __restrict__ agg, const float* __restrict__ m_in,
                               const float* __restrict__ invl_in, const float* __restrict__ d_agg,
                               const int32_t* __restrict__ num_chunks_ptr, const HubChunk* __restrict__ chunks,
                               float2* __restrict__ ecoef, float* __restrict__ partial /* [chunks][DIM] */) {
  using G = RowGeom<DIM>;
  using H = HubGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN, NG = H::NG, PER = H::PER;
  constexpr int HEADS = DIM / HEAD_DIM;
  __shared__ __align__(16) float q_s[DIM];
  __shared__ __align__(16) float dag_s[DIM];
  __shared__ __align__(16) float part_s[NG * DIM];
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int group = (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
  const int num_chunks = *num_chunks_ptr;
  for (int c = blockIdx.x; c < num_chunks; c += gridDim.x) {
    const HubChunk ch = chunks[c];
    const int64_t nrow = ch.node;
    // query and d_agg rows of the hub destination, staged once for the CTA
    for (int i = threadIdx.x; i < DIM / 4; i += kThreads) {
      st4(q_s + 4 * i, ldg4(qkvs + nrow * 4 * DIM + 4 * i));
      st4(dag_s + 4 * i, ldg4(d_agg + nrow * DIM + 4 * i));
    }
    __syncthreads();
    float4 q[V], dag[V], ag[V];
    load_row<DIM>(agg + nrow * DIM, lig, ag);
    float delta[V], mh[V], il[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      q[v] = ld4(q_s + 4 * (v * LPN + lig));
      dag[v] = ld4(dag_s + 4 * (v * LPN + lig));
      delta[v] = dot4(dag[v], ag[v]);
      const int h = head_of<DIM, HEAD_DIM>(v, lig);
      mh[v] = m_in[nrow * HEADS + h];
      il[v] = invl_in[nrow * HEADS + h];
    }
    head_reduce<DIM, HEAD_DIM>(delta);
    const int b = min(group * PER, ch.edge_count);
    const int cnt = min(PER, ch.edge_count - b);
    int cnt_max = cnt;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt_max = max(cnt_max, __shfl_xor_sync(0xffffffffu, cnt_max, off));
    float4 dq[V];
#pragma unroll
    for (int v = 0; v < V; ++v) dq[v] = zero4();
    bwd_dst_edges_serial<DIM, HEAD_DIM, kEdgeUnroll>(qkvs, q, dag, delta, mh, il, col, eperm, alpha_mask, ch.edge_begin + b,
                                                     cnt, cnt_max, nrow, lig, ecoef, dq);
#pragma unroll
    for (int v = 0; v < V; ++v) st4(part_s + group * DIM + 4 * (v * LPN + lig), dq[v]);
    __syncthreads();
    if (threadIdx.x < DIM / 4) {   // lane groups added in group order
      float4 s = zero4();
      for (int g = 0; g < NG; ++g) s = add4(s, ld4(part_s + g * DIM + 4 * threadIdx.x));
      st4(partial + (int64_t)c * DIM + 4 * threadIdx.x, s);
    }
    __syncthreads();
  }
}

// Sums the chunk partials of every hub row (chunk order), stores the gradient rows, and — when asked — writes this
// CTA's column sums of those rows as one partial row for the caller's fixed-order column reduction.
// ROWS = 1: d_query (destination hubs); ROWS = 2: d_key | d_value (source hubs).
template <int DIM, int ROWS>
__global__ void __launch_bounds__(kThreads)
tconv_bwd_hub_combine_kernel(const int32_t* __restrict__ num_rows_ptr, const HubRow* __restrict__ rows,
                             const float* __restrict__ partial /* [chunks][ROWS*DIM] */, float* __restrict__ d_qkvs,
                             __nv_bfloat16* __restrict__ d_hi, __nv_bfloat16* __restrict__ d_lo, int block_offset,
                             float* __restrict__ colsum_rows /* [gridDim.x][width] or NULL */, int width,
                             int col_offset) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN, NG = HubGeom<DIM>::NG;
  __shared__ __align__(16) float sum_s[NG * ROWS * DIM];
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int group = (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
  const int num_rows = *num_rows_ptr;
  float4 colsum[ROWS][V];
#pragma unroll
  for (int r = 0; r < ROWS; ++r)
#pragma unroll
    for (int v = 0; v < V; ++v) colsum[r][v] = zero4();
  for (int slot = blockIdx.x * NG + group; slot < num_rows; slot += gridDim.x * NG) {
    const HubRow hub = rows[slot];
    float4 s[ROWS][V];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int v = 0; v < V; ++v) s[r][v] = zero4();
    constexpr int kAhead = 4;   // chunk partials loaded ahead of the (ordered) sum
    for (int c0 = 0; c0 < hub.num_chunks; c0 += kAhead) {
      float4 part[kAhead][ROWS][V];
#pragma unroll
      for (int u = 0; u < kAhead; ++u) {
        const int c = min(c0 + u, hub.num_chunks - 1);
        const float* src = partial + (int64_t)(hub.first_chunk + c) * ROWS * DIM;
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
          for (int v = 0; v < V; ++v) part[u][r][v] = ldg4(src + r * DIM + 4 * (v * LPN + lig));
      }
#pragma unroll
      for (int u = 0; u < kAhead; ++u) {
        if (c0 + u >= hub.num_chunks) break;
#pragma unroll
        for (int r = 0; r < ROWS; ++r)
#pragma unroll
          for (int v = 0; v < V; ++v) s[r][v] = add4(s[r][v], part[u][r][v]);
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int v = 0; v < V; ++v) {
        store_grad4(d_qkvs, d_hi, d_lo, (int64_t)hub.node * 4 * DIM + (block_offset + r) * DIM + 4 * (v * LPN + lig),
                    s[r][v]);
        colsum[r][v] = add4(colsum[r][v], s[r][v]);
      }
  }
  if (colsum_rows == nullptr) return;
#pragma unroll
  for (int r = 0; r < ROWS; ++r)
#pragma unroll
    for (int v = 0; v < V; ++v) st4(sum_s + (group * ROWS + r) * DIM + 4 * (v * LPN + lig), colsum[r][v]);
  __syncthreads();
  float* mine = colsum_rows + (size_t)blockIdx.x * width;
  for (int i = threadIdx.x; i < width; i += kThreads) {
    float t = 0.f;
    if (i >= col_offset && i < col_offset + ROWS * DIM)
      for (int g = 0; g < NG; ++g) t += sum_s[g * ROWS * DIM + (i - col_offset)];
    mine[i] = t;   // the columns that are not ours are zero: the row joins the caller's partial rows as it is
  }
}

// ------------------------------------------------------------------------------- backward, source side
template <int DIM, int HEAD_DIM>
__global__ void __launch_bounds__(kThreads, 2)
tconv_bwd_src_hub_chunk_kernel(const float* __restrict__ qkvs, const int32_t* __restrict__ row,
                               const int32_t* __restrict__ cpos, const float* __restrict__ d_agg,
                               const float2* __restrict__ ecoef, const int32_t* __restrict__ num_chunks_ptr,
                               const HubChunk* __restrict__ chunks, float* __restrict__ partial /* [chunks][2*DIM] */) {
  using G = RowGeom<DIM>;
  using H = HubGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN, NG = H::NG, PER = H::PER;
  __shared__ __align__(16) float part_s[NG * 2 * DIM];
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int group = (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
  const int num_chunks = *num_chunks_ptr;
  for (int c = blockIdx.x; c < num_chunks; c += gridDim.x) {
    const HubChunk ch = chunks[c];
    const int b = min(group * PER, ch.edge_count);
    const int cnt = min(PER, ch.edge_count - b);
    float4 dk[V], dv[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { dk[v] = zero4(); dv[v] = zero4(); }
    bwd_src_edges_serial<DIM, HEAD_DIM>(qkvs, d_agg, ecoef, row, cpos, ch.edge_begin + b, ch.edge_begin + b + cnt, lig,
                                        dk, dv);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      st4(part_s + group * 2 * DIM + 4 * (v * LPN + lig), dk[v]);
      st4(part_s + group * 2 * DIM + DIM + 4 * (v * LPN + lig), dv[v]);
    }
    __syncthreads();
    for (int f = threadIdx.x; f < 2 * DIM / 4; f += kThreads) {   // lane groups added in group order
      float4 s = zero4();
      for (int g = 0; g < NG; ++g) s = add4(s, ld4(part_s + g * 2 * DIM + 4 * f));
      st4(partial + (int64_t)c * 2 * DIM + 4 * f, s);
    }
    __syncthreads();
  }
}

int chunk_grid(int64_t num_edges) {
  // the number of chunks is device data: a persistent grid of at most two CTAs per SM strides over them
  const int64_t cap = hub_cap_chunks(num_edges);
  return (int)(cap < 2 * kNumSMs ? cap : 2 * kNumSMs);
}

}  // namespace

int tconv_fwd_hubs(const float* qkvs, int dim, int heads, const int32_t* col, const int32_t* eperm, int64_t num_edges,
                   const float* w_beta, const float* alpha_mask, float* out, float* agg, float* beta, float* m,
                   float* inv_l, const void* hub_plan, void* hub_ws, double* stat_rows, cudaStream_t stream) {
  const HubPlanView plan = hub_plan_view(const_cast<void*>(hub_plan), num_edges);
  float* partial = static_cast<float*>(hub_ws);
  const int grid = chunk_grid(num_edges);
#define CALL(D, C)                                                                                                   \
  {                                                                                                                  \
    tconv_fwd_hub_chunk_kernel<D, C><<<grid, kThreads, 0, stream>>>(qkvs, col, eperm, alpha_mask, plan.counts + 1,  \
                                                                    plan.dst_chunks, partial);                      \
    const size_t smem = stat_rows ? (size_t)HubGeom<D>::NG * 2 * D * sizeof(double) : 0;                            \
    tconv_fwd_hub_combine_kernel<D, C><<<kHubColsumCtas, kThreads, smem, stream>>>(                                 \
        qkvs, plan.counts, plan.dst_rows, partial, w_beta, out, agg, beta, m, inv_l, stat_rows);                    \
  }
  ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("tconv_fwd_hub");
  count_launch();
  return ETPGT_OK;
}

int tconv_bwd_dst_hubs(const float* qkvs, int dim, int heads, const int32_t* col, const int32_t* eperm,
                       int64_t num_edges, const float* alpha_mask, const float* agg, const float* m, const float* inv_l,
                       const float* d_agg, float2* ecoef, float* d_qkvs, __nv_bfloat16* d_hi, __nv_bfloat16* d_lo,
                       float* colsum_rows, int width, int col_offset, const void* hub_plan, void* hub_ws,
                       cudaStream_t stream) {
  const HubPlanView plan = hub_plan_view(const_cast<void*>(hub_plan), num_edges);
  float* partial = static_cast<float*>(hub_ws);
  const int grid = chunk_grid(num_edges);
#define CALL(D, C)                                                                                                   \
  {                                                                                                                  \
    tconv_bwd_dst_hub_chunk_kernel<D, C><<<grid, kThreads, 0, stream>>>(qkvs, col, eperm, alpha_mask, agg, m, inv_l, \
                                                                        d_agg, plan.counts + 1, plan.dst_chunks,    \
                                                                        ecoef, partial);                            \
    tconv_bwd_hub_combine_kernel<D, 1><<<kHubColsumCtas, kThreads, 0, stream>>>(                                    \
        plan.counts, plan.dst_rows, partial, d_qkvs, d_hi, d_lo, 0, colsum_rows, width, col_offset);                \
  }
  ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("tconv_bwd_dst_hub");
  count_launch();
  return ETPGT_OK;
}

int tconv_bwd_src_hubs(const float* qkvs, int dim, int heads, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                       const float* d_agg, const float2* ecoef, float* d_qkvs, __nv_bfloat16* d_hi, __nv_bfloat16* d_lo,
                       float* colsum_rows, const void* hub_plan, void* hub_ws, cudaStream_t stream) {
  const HubPlanView plan = hub_plan_view(const_cast<void*>(hub_plan), num_edges);
  float* partial = static_cast<float*>(hub_ws);
  const int grid = chunk_grid(num_edges);
#define CALL(D, C)                                                                                                   \
  {                                                                                                                  \
    tconv_bwd_src_hub_chunk_kernel<D, C><<<grid, kThreads, 0, stream>>>(qkvs, row, cpos, d_agg, ecoef,              \
                                                                        plan.counts + 3, plan.src_chunks, partial); \
    tconv_bwd_hub_combine_kernel<D, 2><<<kHubColsumCtas, kThreads, 0, stream>>>(                                    \
        plan.counts + 2, plan.src_rows, partial, d_qkvs, d_hi, d_lo, 1, colsum_rows, 2 * D, 0);                     \
  }
  ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("tconv_bwd_src_hub");
  count_launch();
  return ETPGT_OK;
}

}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_hub_plan_bytes(int64_t num_edges) { return hub_plan_bytes(num_edges < 0 ? 0 : num_edges); }

extern "C" size_t etpgt_hub_plan_workspace_bytes(int64_t num_nodes) {
  size_t temp = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, temp, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                (int)(num_nodes > 0 ? num_nodes : 1));
  return 2 * align_up((size_t)(num_nodes > 0 ? num_nodes : 1) * sizeof(unsigned long long)) + align_up(temp) + 256;
}

extern "C" int etpgt_hub_plan(const int32_t* rowptr, const int32_t* colptr, int64_t num_nodes, int64_t num_edges,
                              void* plan_, void* ws, size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_nodes >= 0 && num_edges >= 0 && num_nodes < (int64_t(1) << 31), "hub_plan: bad sizes");
  ETPGT_REQUIRE(rowptr && colptr && plan_, "hub_plan: null pointer");
  if (ws_bytes < etpgt_hub_plan_workspace_bytes(num_nodes)) {
    set_error("hub_plan: workspace %zu < %zu", ws_bytes, etpgt_hub_plan_workspace_bytes(num_nodes));
    return ETPGT_EWORKSPACE;
  }
  const HubPlanView plan = hub_plan_view(plan_, num_edges);
  cudaMemsetAsync(plan.counts, 0, 4 * sizeof(int32_t), stream);
  if (num_nodes == 0) return ETPGT_OK;
  Workspace w(ws, ws_bytes);
  unsigned long long* val = w.take<unsigned long long>((size_t)num_nodes);
  unsigned long long* offset = w.take<unsigned long long>((size_t)num_nodes);
  size_t temp_bytes = ws_bytes - w.used;
  void* temp = w.base + w.used;
  const int grid = grid_for(num_nodes, 256, 8);
  for (int side = 0; side < 2; ++side) {
    const int32_t* ptr = side == 0 ? rowptr : colptr;
    hub_flags_kernel<<<grid, 256, 0, stream>>>(ptr, num_nodes, val);
    ETPGT_CHECK_LAUNCH("hub_flags");
    cudaError_t e = cub::DeviceScan::ExclusiveSum(temp, temp_bytes, val, offset, (int)num_nodes, stream);
    if (e != cudaSuccess) {
      set_error("hub_plan: scan failed: %s", cudaGetErrorString(e));
      return ETPGT_ECUDA;
    }
    count_launch();
    hub_emit_kernel<<<grid, 256, 0, stream>>>(ptr, num_nodes, val, offset, side == 0 ? plan.dst_rows : plan.src_rows,
                                              side == 0 ? plan.dst_chunks : plan.src_chunks, plan.counts + 2 * side);
    ETPGT_CHECK_LAUNCH("hub_emit");
  }
  return ETPGT_OK;
}
