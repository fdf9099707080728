// a5: fused TransformerConv over the destination-sorted CSR (forward) and CSR + CSC (backward).
// PyG TransformerConv(concat=True, beta=True, root_weight=True) as reached from
// etpgt/model/graph_transformer.py:73-98,174 (semantics: SURVEY.md §3.3 / oracle/conv_ref.py).
//
// Layout: qkvs [N, 4*DIM] row-major = query | key | value | skip, so the key and value rows an
// edge gathers are one contiguous 2*DIM*4-byte span.  A lane group of LPN = min(32, DIM/4)
// lanes owns one destination row; each lane keeps V = DIM/(4*LPN) float4 of it, and the
// per-head dot products are butterfly reductions over the lanes of that head (head_reduce).
// Softmax is one-pass (running max / running sum, flash-style) so every key/value row is read
// exactly once; logits, alphas and the [E, DIM] gathers of the PyG path never exist in HBM.
//
// HBM-bound.  Algorithmic bytes (fp32): forward 2*DIM*4 per edge + 4*DIM*4 per node
// (q, skip in; out, agg out); backward 4*DIM*4 per edge + 10*DIM*4 per node (DESIGN.md).
#include <cuda_bf16.h>
#include <math.h>

#include <limits.h>

#include "tconv.cuh"

#define TRY_RC(expr)                   \
  do {                                 \
    int rc__ = (expr);                 \
    if (rc__ != ETPGT_OK) return rc__; \
  } while (0)

namespace etpgt {
namespace {

// Edges per unroll group of the session-batch (sparse) variants
template <int DIM>
constexpr int kSparseUnroll = RowGeom<DIM>::V > 1 ? 1 : 2;

// [begin, begin + deg) = the edge range of `node` in ptr (rowptr or colptr); deg = 0 past the last node
__device__ __forceinline__ void node_range(const int32_t* __restrict__ ptr, int64_t node, int64_t num_nodes, int& begin,
                                           int& deg) {
  begin = 0;
  deg = 0;
  if (node < num_nodes) {
    begin = ptr[node];
    deg = ptr[node + 1] - begin;
  }
}

// ------------------------------------------------------------------------------- forward
// (measured on the 32,768-session batch, dim 256: four resident CTAs per SM — 64 registers — run the sparse variant
// 12 % faster than three; the backward kernels lose more to spills than they gain from a fourth CTA)
template <int DIM, int HEAD_DIM, int UNROLL>
__global__ void __launch_bounds__(kThreads, UNROLL <= 2 ? 4 : 2)
tconv_fwd_kernel(const float* __restrict__ qkvs, int64_t num_nodes, const int32_t* __restrict__ rowptr,
                 const int32_t* __restrict__ col, const int32_t* __restrict__ eperm,
                 const float* __restrict__ w_beta, const float* __restrict__ alpha_mask,
                 float* __restrict__ out, float* __restrict__ agg_out, float* __restrict__ beta_out,
                 float* __restrict__ m_out, float* __restrict__ invl_out, int hub_threshold) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t warp_global = (blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5;
  const int64_t node = warp_global * G::GROUPS + lane / LPN;
  const bool valid = node < num_nodes;
  if (warp_global * G::GROUPS >= num_nodes) return;  // whole warp out of range

  const int64_t nrow = valid ? node : 0;
  const float* self = qkvs + nrow * 4 * DIM;
  int begin, deg;
  node_range(rowptr, node, num_nodes, begin, deg);
  float4 q[V], xr[V];
  load_row<DIM>(self, lig, q);
  load_row<DIM>(self + 3 * DIM, lig, xr);
  const bool hub = deg > hub_threshold;   // cut into chunks by the hub kernels (tconv_hub.cu), skipped here
  if (hub) deg = 0;
  const EdgeMeta meta = load_edge_meta(col, alpha_mask != nullptr ? eperm : nullptr, begin, deg, 0, lig);
  int deg_max = deg;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) deg_max = max(deg_max, __shfl_xor_sync(0xffffffffu, deg_max, off));

  float m[V], l[V];
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) { m[v] = -INFINITY; l[v] = 0.f; acc[v] = zero4(); }
  fwd_edges<DIM, HEAD_DIM, UNROLL>(qkvs, q, col, eperm, alpha_mask, begin, deg, deg_max, nrow, lig, meta, m, l, acc);
  fwd_epilogue<DIM, HEAD_DIM>(xr, valid && !hub, nrow, lig, m, l, acc, w_beta, out, agg_out, beta_out, m_out,
                              invl_out);
}

// The same forward as a persistent kernel that also takes the BatchNorm statistics of its output (column sums of
// out and out^2 in double) while the rows are in registers: the layer's separate statistics pass — one more read of
// [N, DIM] — disappears.  Lane groups accumulate into their own shared-memory slots, the CTA's groups are added in a
// fixed order into one partial row, a second stage adds the rows in a fixed order: deterministic, no atomics.
template <int DIM, int HEAD_DIM, int UNROLL>
__global__ void __launch_bounds__(kThreads, UNROLL <= 2 ? 4 : 2)
tconv_fwd_stats_kernel(const float* __restrict__ qkvs, int64_t num_nodes, const int32_t* __restrict__ rowptr,
                       const int32_t* __restrict__ col, const int32_t* __restrict__ eperm,
                       const float* __restrict__ w_beta, const float* __restrict__ alpha_mask,
                       float* __restrict__ out, float* __restrict__ agg_out, float* __restrict__ beta_out,
                       float* __restrict__ m_out, float* __restrict__ invl_out, int hub_threshold,
                       double* __restrict__ stat_partial /* [gridDim.x][2*DIM] */) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  extern __shared__ double stat_s[];   // [(kThreads/32)*GROUPS][2*DIM]
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int warp_in_cta = threadIdx.x >> 5;
  const int64_t nodes_per_cta = (kThreads / 32) * G::GROUPS;
  double* stat_mine = stat_s + (size_t)(warp_in_cta * G::GROUPS + lane / LPN) * 2 * DIM;
#pragma unroll
  for (int v = 0; v < V; ++v)
#pragma unroll
    for (int c = 0; c < 4; ++c) { stat_mine[4 * (v * LPN + lig) + c] = 0.0; stat_mine[DIM + 4 * (v * LPN + lig) + c] = 0.0; }
  // Each warp walks its nodes one ahead: the next node's edge range is loaded at the top of an iteration and the
  // first chunk of its edge metadata after this node's edges, so neither waits on the other's loads.
  const int64_t stride = (int64_t)gridDim.x * nodes_per_cta;
  const int32_t* ep = alpha_mask != nullptr ? eperm : nullptr;
  // deg = -1: a hub row (cut into chunks by the hub kernels, tconv_hub.cu, skipped here); the edge walk takes it as a
  // row without edges
  int begin, deg;
  node_range(rowptr, blockIdx.x * nodes_per_cta + warp_in_cta * G::GROUPS + lane / LPN, num_nodes, begin, deg);
  if (deg > hub_threshold) deg = -1;
  EdgeMeta meta = load_edge_meta(col, ep, begin, deg, 0, lig);
  for (int64_t base = blockIdx.x * nodes_per_cta; base < num_nodes; base += stride) {
    const int64_t warp_base = base + warp_in_cta * G::GROUPS;
    if (warp_base >= num_nodes) continue;  // warp-uniform
    const int64_t node = warp_base + lane / LPN;
    const bool valid = node < num_nodes;
    const int64_t nrow = valid ? node : 0;
    const float* self = qkvs + nrow * 4 * DIM;
    float4 q[V];
    load_row<DIM>(self, lig, q);
    int next_begin, next_deg;
    node_range(rowptr, node + stride, num_nodes, next_begin, next_deg);
    if (next_deg > hub_threshold) next_deg = -1;
    int deg_max = deg;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) deg_max = max(deg_max, __shfl_xor_sync(0xffffffffu, deg_max, off));
    float m[V], l[V];
    float4 acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { m[v] = -INFINITY; l[v] = 0.f; acc[v] = zero4(); }
    fwd_edges<DIM, HEAD_DIM, UNROLL>(qkvs, q, col, eperm, alpha_mask, begin, deg, deg_max, nrow, lig, meta, m, l, acc);
    meta = load_edge_meta(col, ep, next_begin, next_deg, 0, lig);
    float4 xr[V];
    load_row<DIM>(self + 3 * DIM, lig, xr);
    fwd_epilogue<DIM, HEAD_DIM>(xr, valid && deg >= 0, nrow, lig, m, l, acc, w_beta, out, agg_out, beta_out, m_out,
                                invl_out, stat_mine);
    begin = next_begin;
    deg = next_deg;
  }
  stats_flush<DIM>(stat_s, stat_partial + (size_t)blockIdx.x * 2 * DIM);
}

// one warp per output column: lanes stride over the partial rows, fixed butterfly -> deterministic
__global__ void stats_reduce_kernel(const double* __restrict__ partial, int parts, int width, double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= width) return;
  double s = 0;
  for (int p = lane; p < parts; p += 32) s += partial[(int64_t)p * width + i];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if (lane == 0) out[i] = s;
}

// ------------------------------------------------------------ backward, destination pass
// LANES (session batches): edge metadata in lanes, nodes walked one ahead; else (dense graphs) the serial walk over
// 4-edge groups, each node's edge range loaded in its own iteration (the lane walk measured slower there).
// Per destination i: gate backward (d_agg, d_skip, w_beta partials), delta_h = <d_agg, agg>_h,
// then over in-edges: alpha (recomputed from saved m, 1/l), d_alpha = <d_agg, v_j>_h,
// d_logit = alpha (d_alpha*mask - delta), d_query += scale*d_logit*k_j.  Emits per-edge
// (alpha*mask, scale*d_logit) for the source pass.
template <int DIM, int HEAD_DIM, bool LANES, bool COLSUM>
__global__ void __launch_bounds__(kThreads, LANES ? 3 : 2)
tconv_bwd_dst_kernel(const float* __restrict__ qkvs, const float* __restrict__ d_out, int64_t num_nodes,
                     const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                     const int32_t* __restrict__ eperm, const float* __restrict__ w_beta,
                     const float* __restrict__ alpha_mask, const float* __restrict__ agg,
                     const float* __restrict__ beta, const float* __restrict__ m_in,
                     const float* __restrict__ invl_in, float* __restrict__ d_qkvs,
                     __nv_bfloat16* __restrict__ d_hi, __nv_bfloat16* __restrict__ d_lo,
                     float* __restrict__ d_agg_out, float2* __restrict__ ecoef,
                     float* __restrict__ partial /* [grid][(w_beta ? 3 : 0) + (COLSUM ? 2 : 0)][DIM] */,
                     int hub_threshold) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  constexpr int HEADS = DIM / HEAD_DIM;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int warp_in_cta = threadIdx.x >> 5;
  const int64_t nodes_per_cta = (kThreads / 32) * G::GROUPS;

  // Per-group running sums live in shared memory (each lane owns its own float4 slots, so no
  // synchronisation is needed until the final cross-group reduction): [sum dz*agg | sum dz*skip | (their
  // difference, formed at the end)] for the w_beta gradient, then [sum d_query | sum d_skip] for the bias
  // gradients.  Keeping them out of registers lets three CTAs share an SM instead of two.
  extern __shared__ float dyn[];  // [(kThreads/32)*GROUPS][width]
  const int wb = w_beta != nullptr ? 3 : 0, width = (wb + (COLSUM ? 2 : 0)) * DIM;
  float* mine = dyn + (size_t)(warp_in_cta * G::GROUPS + lane / LPN) * width;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int f = v * LPN + lig;
    if (wb) { st4(mine + 4 * f, zero4()); st4(mine + DIM + 4 * f, zero4()); }
    if (COLSUM) { st4(mine + wb * DIM + 4 * f, zero4()); st4(mine + (wb + 1) * DIM + 4 * f, zero4()); }
  }

  constexpr int UNROLL = LANES ? kSparseUnroll<DIM> : kEdgeUnroll;
  const int64_t stride = (int64_t)gridDim.x * nodes_per_cta;
  const int32_t* ep = alpha_mask != nullptr ? eperm : nullptr;
  // deg = -1: a hub row (edges, d_query and its column sums: the hub kernels, tconv_hub.cu); the edge walks take it
  // as a row without edges
  int begin = 0, deg = 0;
  EdgeMeta meta{0, 0};
  if constexpr (LANES) {
    node_range(rowptr, blockIdx.x * nodes_per_cta + warp_in_cta * G::GROUPS + lane / LPN, num_nodes, begin, deg);
    if (deg > hub_threshold) deg = -1;
    meta = load_edge_meta(col, ep, begin, deg, 0, lig);
  }
  for (int64_t base = blockIdx.x * nodes_per_cta; base < num_nodes; base += stride) {
    const int64_t warp_base = base + warp_in_cta * G::GROUPS;
    if (warp_base >= num_nodes) continue;  // warp-uniform
    const int64_t node = warp_base + lane / LPN;
    const bool valid = node < num_nodes;
    const int64_t nrow = valid ? node : 0;
    const float* self = qkvs + nrow * 4 * DIM;

    float4 g[V], xr[V], ag[V], dag[V], q[V];
    load_row<DIM>(d_out + nrow * DIM, lig, g);
    load_row<DIM>(self + 3 * DIM, lig, xr);
    load_row<DIM>(agg + nrow * DIM, lig, ag);
    load_row<DIM>(self, lig, q);
    int next_begin = 0, next_deg = 0;
    if constexpr (LANES) {
      node_range(rowptr, node + stride, num_nodes, next_begin, next_deg);
    } else {
      node_range(rowptr, node, num_nodes, begin, deg);
      if (deg > hub_threshold) deg = -1;
    }
    if (next_deg > hub_threshold) next_deg = -1;
    if (w_beta != nullptr) {
      const float b = beta[nrow];
      float part = 0.f;
#pragma unroll
      for (int v = 0; v < V; ++v) part += dot4(g[v], sub4(xr[v], ag[v]));
      const float dz = group_sum<LPN>(part) * b * (1.f - b);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int f = v * LPN + lig;
        const float4 w1 = ldg4(w_beta + 4 * f), w2 = ldg4(w_beta + DIM + 4 * f), w3 = ldg4(w_beta + 2 * DIM + 4 * f);
        dag[v] = fma4(dz, add4(w1, w3), scale4(1.f - b, g[v]));
        const float4 dxr = fma4(dz, sub4(w2, w3), scale4(b, g[v]));
        if (valid) {
          store_grad4(d_qkvs, d_hi, d_lo, nrow * 4 * DIM + 3 * DIM + 4 * f, dxr);
          st4(mine + 4 * f, fma4(dz, ag[v], ld4(mine + 4 * f)));
          st4(mine + DIM + 4 * f, fma4(dz, xr[v], ld4(mine + DIM + 4 * f)));
          if (COLSUM) st4(mine + (wb + 1) * DIM + 4 * f, add4(ld4(mine + (wb + 1) * DIM + 4 * f), dxr));
        }
      }
    } else {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        dag[v] = g[v];
        if (valid) {
          store_grad4(d_qkvs, d_hi, d_lo, nrow * 4 * DIM + 3 * DIM + 4 * (v * LPN + lig), g[v]);
          if (COLSUM) {
            float* slot = mine + (wb + 1) * DIM + 4 * (v * LPN + lig);
            st4(slot, add4(ld4(slot), g[v]));
          }
        }
      }
    }
    float delta[V], mh[V], il[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
      delta[v] = dot4(dag[v], ag[v]);
      const int h = head_of<DIM, HEAD_DIM>(v, lig);
      mh[v] = m_in[nrow * HEADS + h];
      il[v] = invl_in[nrow * HEADS + h];
      if (valid) st4(d_agg_out + nrow * DIM + 4 * (v * LPN + lig), dag[v]);
    }
    head_reduce<DIM, HEAD_DIM>(delta);

    int deg_max = deg;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) deg_max = max(deg_max, __shfl_xor_sync(0xffffffffu, deg_max, off));
    float4 dq[V];
#pragma unroll
    for (int v = 0; v < V; ++v) dq[v] = zero4();
    if constexpr (!LANES) {
      bwd_dst_edges_serial<DIM, HEAD_DIM, UNROLL>(qkvs, q, dag, delta, mh, il, col, eperm, alpha_mask, begin, deg, deg_max,
                                                  nrow, lig, ecoef, dq);
    } else {
      bwd_dst_edges<DIM, HEAD_DIM, UNROLL>(qkvs, q, dag, delta, mh, il, col, eperm, alpha_mask, begin, deg, deg_max, nrow,
                                           lig, meta, ecoef, dq);
      meta = load_edge_meta(col, ep, next_begin, next_deg, 0, lig);
    }
    if (valid && deg >= 0) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        store_grad4(d_qkvs, d_hi, d_lo, nrow * 4 * DIM + 4 * (v * LPN + lig), dq[v]);
        if (COLSUM) {
          float* slot = mine + wb * DIM + 4 * (v * LPN + lig);
          st4(slot, add4(ld4(slot), dq[v]));
        }
      }
    }
    if constexpr (LANES) {
      begin = next_begin;
      deg = next_deg;
    }
  }

  if (width > 0) {
    // fixed-order reduction of the per-group sums of this CTA
    if (wb) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int f = v * LPN + lig;
        st4(mine + 2 * DIM + 4 * f, sub4(ld4(mine + 4 * f), ld4(mine + DIM + 4 * f)));
      }
    }
    __syncthreads();
    constexpr int NG = (kThreads / 32) * G::GROUPS;
    for (int i = threadIdx.x; i < width; i += kThreads) {
      float s = 0.f;
      for (int gidx = 0; gidx < NG; ++gidx) s += dyn[(size_t)gidx * width + i];
      partial[(int64_t)blockIdx.x * width + i] = s;
    }
  }
}

// Column i of the per-CTA partials goes to out_a[i] when i < width_a, else to
// out_b[off_b0 + (i - width_a)] for the first `dim` of them and out_b[off_b1 + ...] for the next `dim`
// (the two bias-gradient blocks of a pass sit at different offsets of the [4*dim] bias gradient).
constexpr int kReduceWarps = 32;
__global__ void __launch_bounds__(kReduceWarps * 32)
reduce_partials_kernel(const float* __restrict__ partial, int parts, int width, int width_a,
                       float* __restrict__ out_a, float* __restrict__ out_b, int dim, int off_b0, int off_b1) {
  // A CTA owns 32 consecutive columns: lane = column (every load is one coalesced 128-byte row
  // segment), warp w adds parts w, w+32, ... with eight loads in flight (up to 1,184 partials: five
  // dependent rounds per warp), the 32 warp sums are then added in warp order -> deterministic.
  __shared__ float warp_sum[kReduceWarps][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  float s = 0.f;
  if (i < width) {
    int p = w;
    for (; p + 7 * kReduceWarps < parts; p += 8 * kReduceWarps) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = partial[(int64_t)(p + kReduceWarps * u) * width + i];
#pragma unroll
      for (int u = 0; u < 8; ++u) s += v[u];
    }
    for (; p < parts; p += kReduceWarps) s += partial[(int64_t)p * width + i];
  }
  warp_sum[w][lane] = s;
  __syncthreads();
  if (w != 0 || i >= width) return;
  float t = 0.f;
#pragma unroll
  for (int q = 0; q < kReduceWarps; ++q) t += warp_sum[q][lane];
  if (i < width_a) out_a[i] = t;
  else if (i - width_a < dim) out_b[off_b0 + (i - width_a)] = t;
  else out_b[off_b1 + (i - width_a - dim)] = t;
}

// ------------------------------------------------------------------ backward, source pass
// Per source j over its out-edges (CSC): d_key_j += scale*d_logit_e * q_i, d_value_j +=
// alpha_e*mask_e * d_agg_i.  One owner group per row, ascending CSC order: deterministic.
// LANES (session batches): edge metadata in lanes, nodes walked one ahead; else (dense graphs) each lane group walks
// its own edges with the serial source walk, loading its node's edge range in the node's own iteration.
template <int DIM, int HEAD_DIM, bool LANES, bool COLSUM>
__global__ void __launch_bounds__(kThreads, COLSUM ? 3 : 4)
tconv_bwd_src_kernel(const float* __restrict__ qkvs, int64_t num_nodes, const int32_t* __restrict__ colptr,
                     const int32_t* __restrict__ row, const int32_t* __restrict__ cpos,
                     const float* __restrict__ d_agg, const float2* __restrict__ ecoef,
                     float* __restrict__ d_qkvs, __nv_bfloat16* __restrict__ d_hi, __nv_bfloat16* __restrict__ d_lo,
                     float* __restrict__ colsum_partial /* [grid][2*DIM] or NULL */, int hub_threshold) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t nodes_per_cta = (kThreads / 32) * G::GROUPS;
  float4 ck[V], cv[V];   // column sums of d_key / d_value over this CTA's rows (bias gradients)
#pragma unroll
  for (int v = 0; v < V; ++v) { ck[v] = zero4(); cv[v] = zero4(); }
  // the gradient rows of a non-hub source, and their column sums
  auto finish = [&](int64_t node, const float4 (&dk)[V], const float4 (&dv)[V]) {
#pragma unroll
    for (int v = 0; v < V; ++v) {
      store_grad4(d_qkvs, d_hi, d_lo, node * 4 * DIM + DIM + 4 * (v * LPN + lig), dk[v]);
      store_grad4(d_qkvs, d_hi, d_lo, node * 4 * DIM + 2 * DIM + 4 * (v * LPN + lig), dv[v]);
      if (COLSUM) { ck[v] = add4(ck[v], dk[v]); cv[v] = add4(cv[v], dv[v]); }
    }
  };
  // grid-stride over node groups: with the column sums wanted the grid is capped (a few CTAs per SM), so
  // that only a few hundred per-CTA partials have to be reduced afterwards
  const int64_t stride = (int64_t)gridDim.x * nodes_per_cta;
  if constexpr (!LANES) {
    for (int64_t base = blockIdx.x * nodes_per_cta; base < num_nodes; base += stride) {
      const int64_t node = base + (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
      if (node >= num_nodes) continue;
      const int begin = colptr[node], end = colptr[node + 1];
      if (end - begin > hub_threshold) continue;   // a hub source: tconv_hub.cu
      float4 dk[V], dv[V];
#pragma unroll
      for (int v = 0; v < V; ++v) { dk[v] = zero4(); dv[v] = zero4(); }
      bwd_src_edges_serial<DIM, HEAD_DIM>(qkvs, d_agg, ecoef, row, cpos, begin, end, lig, dk, dv);
      finish(node, dk, dv);
    }
  } else {
    int begin, deg;
    node_range(colptr, blockIdx.x * nodes_per_cta + (threadIdx.x >> 5) * G::GROUPS + lane / LPN, num_nodes, begin, deg);
    bool hub = deg > hub_threshold;   // a hub source: tconv_hub.cu
    if (hub) deg = 0;
    EdgeMeta meta = load_edge_meta(row, cpos, begin, deg, 0, lig);
    for (int64_t base = blockIdx.x * nodes_per_cta; base < num_nodes; base += stride) {
      const int64_t warp_base = base + (threadIdx.x >> 5) * G::GROUPS;
      if (warp_base >= num_nodes) continue;  // warp-uniform
      const int64_t node = warp_base + lane / LPN;
      int next_begin, next_deg;
      node_range(colptr, node + stride, num_nodes, next_begin, next_deg);
      const bool next_hub = next_deg > hub_threshold;
      if (next_hub) next_deg = 0;
      int deg_max = deg;
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) deg_max = max(deg_max, __shfl_xor_sync(0xffffffffu, deg_max, off));
      float4 dk[V], dv[V];
#pragma unroll
      for (int v = 0; v < V; ++v) { dk[v] = zero4(); dv[v] = zero4(); }
      bwd_src_edges<DIM, HEAD_DIM, kSparseUnroll<DIM>>(qkvs, d_agg, ecoef, row, cpos, begin, deg, deg_max, lig, meta, dk,
                                                       dv);
      meta = load_edge_meta(row, cpos, next_begin, next_deg, 0, lig);
      if (node < num_nodes && !hub) finish(node, dk, dv);
      begin = next_begin;
      deg = next_deg;
      hub = next_hub;
    }
  }
  if (COLSUM) {
    // groups added in a fixed order -> deterministic
    extern __shared__ float dyn[];  // [(kThreads/32)*GROUPS][2*DIM]
    const int group_in_cta = (threadIdx.x >> 5) * G::GROUPS + lane / LPN;
    float* mine = dyn + (size_t)group_in_cta * 2 * DIM;
#pragma unroll
    for (int v = 0; v < V; ++v) {
      st4(mine + 4 * (v * LPN + lig), ck[v]);
      st4(mine + DIM + 4 * (v * LPN + lig), cv[v]);
    }
    __syncthreads();
    constexpr int NG = (kThreads / 32) * G::GROUPS;
    for (int i = threadIdx.x; i < 2 * DIM; i += kThreads) {
      float s = 0.f;
      for (int gidx = 0; gidx < NG; ++gidx) s += dyn[(size_t)gidx * 2 * DIM + i];
      colsum_partial[(int64_t)blockIdx.x * 2 * DIM + i] = s;
    }
  }
}

// persistent destination pass: as many CTAs as are resident (3 per SM for the sparse variant, 2 for the
// dense one, which then runs two even waves)
int dst_pass_grid(int64_t num_nodes, int nodes_per_cta, bool sparse) {
  return grid_for(num_nodes, nodes_per_cta, sparse ? 3 : 4);
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_tconv_hub_workspace_bytes(int64_t num_edges, int dim) {
  // per-chunk partials: forward (m, l, acc) = dim + 16 floats, backward dst dq = dim, backward src (dk | dv) = 2*dim
  const int row = 2 * dim > dim + 16 ? 2 * dim : dim + 16;
  return align_up((size_t)hub_cap_chunks(num_edges < 0 ? 0 : num_edges) * row * sizeof(float)) + 256;
}

constexpr int kStatCtasPerSm = 4;

extern "C" size_t etpgt_tconv_fwd_bn_workspace_bytes(int dim) {
  return align_up((size_t)(kNumSMs * kStatCtasPerSm + kHubColsumCtas) * 2 * dim * sizeof(double)) + 256;
}

// bn_sums == NULL: the plain forward.  Else the persistent statistics variant: bn_sums [2*dim] doubles = column sums
// of out and of out^2 over all rows (what etpgt_bn_stats computes from a second pass over out).
static int tconv_fwd_impl(const float* qkvs, int64_t num_nodes, int dim, int heads, const int32_t* rowptr,
                          const int32_t* col, const int32_t* eperm, int64_t num_edges, const float* w_beta,
                          const float* alpha_mask, float* out, float* agg, float* beta, float* m, float* inv_l,
                          const void* hub_plan, void* hub_ws, size_t hub_ws_bytes, double* bn_sums, void* bn_ws,
                          size_t bn_ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_nodes >= 0 && num_edges >= 0, "tconv_fwd: negative size");
  ETPGT_REQUIRE(qkvs && rowptr && out && agg && m && inv_l, "tconv_fwd: null pointer");
  ETPGT_REQUIRE(num_edges == 0 || (col && eperm), "tconv_fwd: null edge arrays");
  ETPGT_REQUIRE(w_beta == nullptr || beta != nullptr, "tconv_fwd: beta output required with w_beta");
  ETPGT_REQUIRE(hub_plan == nullptr || (hub_ws != nullptr && hub_ws_bytes >= etpgt_tconv_hub_workspace_bytes(num_edges, dim)),
                "tconv_fwd: hub workspace %zu < %zu", hub_ws_bytes, etpgt_tconv_hub_workspace_bytes(num_edges, dim));
  ETPGT_REQUIRE(bn_sums == nullptr || (bn_ws != nullptr && bn_ws_bytes >= etpgt_tconv_fwd_bn_workspace_bytes(dim)),
                "tconv_fwd_bn: workspace %zu < %zu", bn_ws_bytes, etpgt_tconv_fwd_bn_workspace_bytes(dim));
  if (num_nodes == 0) {
    if (bn_sums != nullptr) cudaMemsetAsync(bn_sums, 0, (size_t)2 * dim * sizeof(double), stream);
    return ETPGT_OK;
  }
  const bool sparse = num_edges < 8 * num_nodes;  // session batches: short rows -> shallower unroll, more warps
  const int hub_threshold = hub_plan != nullptr ? kHubThreshold : INT_MAX;
  double* stat_partial = static_cast<double*>(bn_ws);
  int parts = 0;
#define CALL(D, C)                                                                               \
  {                                                                                              \
    const int64_t npc = (kThreads / 32) * RowGeom<D>::GROUPS;                                    \
    const int64_t grid = (num_nodes + npc - 1) / npc;                                            \
    if (bn_sums != nullptr) {                                                                    \
      parts = grid_for(num_nodes, (int)npc, sparse ? kStatCtasPerSm : 2);                        \
      const size_t smem = (size_t)npc * 2 * D * sizeof(double);                                  \
      if (sparse)                                                                                \
        tconv_fwd_stats_kernel<D, C, kSparseUnroll<D>><<<parts, kThreads, smem, stream>>>(qkvs, num_nodes, rowptr, col, eperm, w_beta, \
                                            alpha_mask, out, agg, beta, m, inv_l, hub_threshold, stat_partial); \
      else                                                                                       \
        tconv_fwd_stats_kernel<D, C, 4><<<parts, kThreads, smem, stream>>>(qkvs, num_nodes, rowptr, col, eperm, w_beta, \
                                            alpha_mask, out, agg, beta, m, inv_l, hub_threshold, stat_partial); \
    } else if (sparse)                                                                           \
      tconv_fwd_kernel<D, C, kSparseUnroll<D>><<<(unsigned)grid, kThreads, 0, stream>>>(qkvs, num_nodes, rowptr, col, eperm,   \
                                                          w_beta, alpha_mask, out, agg, beta, m, inv_l, hub_threshold); \
    else                                                                                         \
      tconv_fwd_kernel<D, C, 4><<<(unsigned)grid, kThreads, 0, stream>>>(qkvs, num_nodes, rowptr, col, eperm,   \
                                                          w_beta, alpha_mask, out, agg, beta, m, inv_l, hub_threshold); \
  }
  ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("tconv_fwd");
  if (hub_plan != nullptr) {
    TRY_RC(tconv_fwd_hubs(qkvs, dim, heads, col, eperm, num_edges, w_beta, alpha_mask, out, agg, beta, m, inv_l, hub_plan,
                          hub_ws, bn_sums ? stat_partial + (size_t)parts * 2 * dim : nullptr, stream));
    if (bn_sums != nullptr) parts += kHubColsumCtas;
  }
  if (bn_sums != nullptr) {
    stats_reduce_kernel<<<(2 * dim * 32 + 255) / 256, 256, 0, stream>>>(stat_partial, parts, 2 * dim, bn_sums);
    ETPGT_CHECK_LAUNCH("tconv_fwd statistics reduce");
  }
  return ETPGT_OK;
}

extern "C" int etpgt_tconv_fwd_hub(const float* qkvs, int64_t num_nodes, int dim, int heads,
                                   const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                                   int64_t num_edges, const float* w_beta, const float* alpha_mask, float* out,
                                   float* agg, float* beta, float* m, float* inv_l, const void* hub_plan,
                                   void* hub_ws, size_t hub_ws_bytes, etpgt_stream_t stream) {
  return tconv_fwd_impl(qkvs, num_nodes, dim, heads, rowptr, col, eperm, num_edges, w_beta, alpha_mask, out, agg, beta, m,
                        inv_l, hub_plan, hub_ws, hub_ws_bytes, nullptr, nullptr, 0, stream);
}

extern "C" int etpgt_tconv_fwd_bn(const float* qkvs, int64_t num_nodes, int dim, int heads, const int32_t* rowptr,
                                  const int32_t* col, const int32_t* eperm, int64_t num_edges, const float* w_beta,
                                  const float* alpha_mask, float* out, float* agg, float* beta, float* m, float* inv_l,
                                  const void* hub_plan, void* hub_ws, size_t hub_ws_bytes, double* bn_sums, void* bn_ws,
                                  size_t bn_ws_bytes, etpgt_stream_t stream) {
  ETPGT_REQUIRE(bn_sums != nullptr, "tconv_fwd_bn: null bn_sums");
  return tconv_fwd_impl(qkvs, num_nodes, dim, heads, rowptr, col, eperm, num_edges, w_beta, alpha_mask, out, agg, beta, m,
                        inv_l, hub_plan, hub_ws, hub_ws_bytes, bn_sums, bn_ws, bn_ws_bytes, stream);
}

extern "C" int etpgt_tconv_fwd(const float* qkvs, int64_t num_nodes, int dim, int heads,
                               const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                               int64_t num_edges, const float* w_beta, const float* alpha_mask, float* out,
                               float* agg, float* beta, float* m, float* inv_l, etpgt_stream_t stream) {
  return etpgt_tconv_fwd_hub(qkvs, num_nodes, dim, heads, rowptr, col, eperm, num_edges, w_beta, alpha_mask, out, agg,
                             beta, m, inv_l, nullptr, nullptr, 0, stream);
}

extern "C" size_t etpgt_tconv_bwd_workspace_bytes(int64_t num_nodes, int64_t num_edges, int dim, int heads) {
  const int64_t src_ctas = 8 * kNumSMs;  // the source pass runs a capped, persistent grid when it sums columns
  return align_up((size_t)num_nodes * dim * sizeof(float)) +
         align_up((size_t)(num_edges > 0 ? num_edges : 1) * heads * sizeof(float2)) +
         align_up((size_t)(kNumSMs * 4 + kHubColsumCtas) * 5 * dim * sizeof(float)) +
         align_up((size_t)(src_ctas + kHubColsumCtas) * 2 * dim * sizeof(float)) + 256;
}

extern "C" int etpgt_tconv_bwd_split_hub(const float* qkvs, const float* d_out, int64_t num_nodes, int dim, int heads,
                                         const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                                         const int32_t* colptr, const int32_t* row, const int32_t* cpos,
                                         int64_t num_edges, const float* w_beta, const float* alpha_mask,
                                         const float* agg, const float* beta, const float* m, const float* inv_l,
                                         float* d_qkvs, void* d_hi_, void* d_lo_, float* d_colsum, float* d_w_beta,
                                         void* ws, size_t ws_bytes, const void* hub_plan, void* hub_ws,
                                         size_t hub_ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(hub_plan == nullptr || (hub_ws != nullptr && hub_ws_bytes >= etpgt_tconv_hub_workspace_bytes(num_edges, dim)),
                "tconv_bwd: hub workspace %zu < %zu", hub_ws_bytes, etpgt_tconv_hub_workspace_bytes(num_edges, dim));
  const int hub_threshold = hub_plan != nullptr ? kHubThreshold : INT_MAX;
  __nv_bfloat16* d_hi = static_cast<__nv_bfloat16*>(d_hi_);
  __nv_bfloat16* d_lo = static_cast<__nv_bfloat16*>(d_lo_);
  ETPGT_REQUIRE(num_nodes >= 0 && num_edges >= 0, "tconv_bwd: negative size");
  ETPGT_REQUIRE(qkvs && d_out && rowptr && colptr && agg && m && inv_l, "tconv_bwd: null pointer");
  ETPGT_REQUIRE((d_hi != nullptr) == (d_lo != nullptr) && (d_hi != nullptr || d_qkvs != nullptr),
                "tconv_bwd: gradient output required: fp32 d_qkvs, or both bf16 parts d_hi / d_lo");
  ETPGT_REQUIRE(w_beta == nullptr || (beta && d_w_beta), "tconv_bwd: beta / d_w_beta required with w_beta");
  if (ws_bytes < etpgt_tconv_bwd_workspace_bytes(num_nodes, num_edges, dim, heads)) {
    set_error("tconv_bwd: workspace %zu < %zu", ws_bytes,
              etpgt_tconv_bwd_workspace_bytes(num_nodes, num_edges, dim, heads));
    return ETPGT_EWORKSPACE;
  }
  if (num_nodes == 0) {
    if (d_colsum != nullptr) cudaMemsetAsync(d_colsum, 0, (size_t)4 * dim * sizeof(float), stream);
    if (d_w_beta != nullptr) cudaMemsetAsync(d_w_beta, 0, (size_t)3 * dim * sizeof(float), stream);
    return ETPGT_OK;
  }
  const bool sparse = num_edges < 8 * num_nodes;  // session batches: short rows -> shallower unroll, more warps
  const int want_colsum = d_colsum != nullptr;
  const int width_a = w_beta ? 3 * dim : 0;
  const int width = width_a + (want_colsum ? 2 * dim : 0);
  Workspace w(ws, ws_bytes);
  float* d_agg = w.take<float>((size_t)num_nodes * dim);
  float2* ecoef = w.take<float2>((size_t)(num_edges > 0 ? num_edges : 1) * heads);
  float* partial = w.take<float>((size_t)(kNumSMs * 4 + kHubColsumCtas) * 5 * dim);
  int grid_a = 1;
#define CALL(D, C)                                                                                   \
  {                                                                                                  \
    const int npc = (kThreads / 32) * RowGeom<D>::GROUPS;                                            \
    grid_a = dst_pass_grid(num_nodes, npc, sparse);                                                        \
    const size_t smem = (size_t)npc * width * sizeof(float);                                         \
    auto kern = sparse ? (want_colsum ? tconv_bwd_dst_kernel<D, C, true, true> : tconv_bwd_dst_kernel<D, C, true, false>) \
                       : (want_colsum ? tconv_bwd_dst_kernel<D, C, false, true> : tconv_bwd_dst_kernel<D, C, false, false>); \
    kern<<<grid_a, kThreads, smem, stream>>>(qkvs, d_out, num_nodes, rowptr, col, eperm, w_beta, alpha_mask, agg,    \
                                             beta, m, inv_l, d_qkvs, d_hi, d_lo, d_agg, ecoef, partial, hub_threshold); \
  }
  ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("tconv_bwd_dst");
  int parts_a = grid_a;
  if (hub_plan != nullptr) {
    // hub destinations: per-edge coefficients and d_query by chunks; their d_query column sums arrive as
    // kHubColsumCtas more partial rows behind the row kernel's
    TRY_RC(tconv_bwd_dst_hubs(qkvs, dim, heads, col, eperm, num_edges, alpha_mask, agg, m, inv_l, d_agg, ecoef, d_qkvs,
                              d_hi, d_lo, want_colsum ? partial + (size_t)grid_a * width : nullptr, width, width_a,
                              hub_plan, hub_ws, stream));
    if (want_colsum) parts_a += kHubColsumCtas;
  }
  if (width > 0) {  // d_w_beta [3*dim]; bias gradients of query -> d_colsum[0:dim], skip -> d_colsum[3*dim:4*dim]
    reduce_partials_kernel<<<(width + 31) / 32, kReduceWarps * 32, 0, stream>>>(partial, parts_a, width, width_a, d_w_beta, d_colsum,
                                                                 dim, 0, 3 * dim);
    ETPGT_CHECK_LAUNCH("tconv dst partial reduce");
  }
  float* src_partial = want_colsum ? w.take<float>((size_t)(8 * kNumSMs + kHubColsumCtas) * 2 * dim) : nullptr;
  int64_t grid_src = 1;
#define CALL(D, C)                                                                                  \
  {                                                                                                 \
    const int64_t npc = (kThreads / 32) * RowGeom<D>::GROUPS;                                       \
    grid_src = (num_nodes + npc - 1) / npc;                                                         \
    if (want_colsum && grid_src > 8 * kNumSMs) grid_src = 8 * kNumSMs;                              \
    const size_t smem = want_colsum ? (size_t)npc * 2 * D * sizeof(float) : 0;                      \
    auto kern = sparse ? (want_colsum ? tconv_bwd_src_kernel<D, C, true, true> : tconv_bwd_src_kernel<D, C, true, false>) \
                       : (want_colsum ? tconv_bwd_src_kernel<D, C, false, true> : tconv_bwd_src_kernel<D, C, false, false>); \
    kern<<<(unsigned)grid_src, kThreads, smem, stream>>>(qkvs, num_nodes, colptr, row, cpos, d_agg, ecoef, d_qkvs, \
                                                         d_hi, d_lo, src_partial, hub_threshold);   \
  }
  ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("tconv_bwd_src");
  int parts_src = (int)grid_src;
  if (hub_plan != nullptr) {
    TRY_RC(tconv_bwd_src_hubs(qkvs, dim, heads, row, cpos, num_edges, d_agg, ecoef, d_qkvs, d_hi, d_lo,
                              want_colsum ? src_partial + (size_t)grid_src * 2 * dim : nullptr, hub_plan, hub_ws, stream));
    if (want_colsum) parts_src += kHubColsumCtas;
  }
  if (want_colsum) {  // key -> d_colsum[dim:2*dim], value -> d_colsum[2*dim:3*dim]
    reduce_partials_kernel<<<(2 * dim + 31) / 32, kReduceWarps * 32, 0, stream>>>(src_partial, parts_src, 2 * dim, 0, nullptr,
                                                                   d_colsum, dim, dim, 2 * dim);
    ETPGT_CHECK_LAUNCH("tconv src colsum reduce");
  }
  return ETPGT_OK;
}

extern "C" int etpgt_tconv_bwd_split(const float* qkvs, const float* d_out, int64_t num_nodes, int dim, int heads,
                                     const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                                     const int32_t* colptr, const int32_t* row, const int32_t* cpos,
                                     int64_t num_edges, const float* w_beta, const float* alpha_mask,
                                     const float* agg, const float* beta, const float* m, const float* inv_l,
                                     float* d_qkvs, void* d_hi, void* d_lo, float* d_colsum, float* d_w_beta,
                                     void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  return etpgt_tconv_bwd_split_hub(qkvs, d_out, num_nodes, dim, heads, rowptr, col, eperm, colptr, row, cpos, num_edges,
                                   w_beta, alpha_mask, agg, beta, m, inv_l, d_qkvs, d_hi, d_lo, d_colsum, d_w_beta, ws,
                                   ws_bytes, nullptr, nullptr, 0, stream);
}

extern "C" int etpgt_tconv_bwd(const float* qkvs, const float* d_out, int64_t num_nodes, int dim, int heads,
                               const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                               const int32_t* colptr, const int32_t* row, const int32_t* cpos,
                               int64_t num_edges, const float* w_beta, const float* alpha_mask,
                               const float* agg, const float* beta, const float* m, const float* inv_l,
                               float* d_qkvs, float* d_w_beta, void* ws, size_t ws_bytes,
                               etpgt_stream_t stream) {
  ETPGT_REQUIRE(d_qkvs != nullptr, "tconv_bwd: null d_qkvs");
  return etpgt_tconv_bwd_split(qkvs, d_out, num_nodes, dim, heads, rowptr, col, eperm, colptr, row, cpos, num_edges,
                               w_beta, alpha_mask, agg, beta, m, inv_l, d_qkvs, nullptr, nullptr, nullptr, d_w_beta,
                               ws, ws_bytes, stream);
}
