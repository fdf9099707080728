// Device helpers shared by the fused TransformerConv kernels (tconv.cu) and their hub-row variants
// (tconv_hub.cu): row loads for the lane-group geometry of common.cuh and the gradient-row store.
#pragma once

#include <cuda_bf16.h>
#include <math.h>

#include "common.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;
constexpr int kEdgeUnroll = 4;
constexpr float kSoftmaxEps = 1e-16f;  // PyG utils.softmax: p / (sum + 1e-16)

template <int DIM>
__device__ __forceinline__ void load_row(const float* __restrict__ row, int lig, float4 (&dst)[RowGeom<DIM>::V]) {
#pragma unroll
  for (int v = 0; v < RowGeom<DIM>::V; ++v) dst[v] = ldg4(row + 4 * (v * RowGeom<DIM>::LPN + lig));
}

// Gradient row store: fp32 (d_qkvs) or, for the tensor-core projection backward, already split as
// x = hi + lo with hi = bf16(x), lo = bf16(x - hi) (what etpgt_split_bf16 would produce from the fp32
// row) so that the [N, 4*DIM] gradient never makes a second trip through HBM.
__device__ __forceinline__ uint2 pack_bf16x4(float a, float b, float c, float d) {
  __nv_bfloat162 p0 = __floats2bfloat162_rn(a, b), p1 = __floats2bfloat162_rn(c, d);
  uint2 r;
  r.x = *reinterpret_cast<uint32_t*>(&p0);
  r.y = *reinterpret_cast<uint32_t*>(&p1);
  return r;
}
__device__ __forceinline__ void store_grad4(float* __restrict__ d_f32, __nv_bfloat16* __restrict__ d_hi,
                                            __nv_bfloat16* __restrict__ d_lo, int64_t offset, float4 g) {
  if (d_hi != nullptr) {
    const float hx = __bfloat162float(__float2bfloat16_rn(g.x)), hy = __bfloat162float(__float2bfloat16_rn(g.y));
    const float hz = __bfloat162float(__float2bfloat16_rn(g.z)), hw = __bfloat162float(__float2bfloat16_rn(g.w));
    *reinterpret_cast<uint2*>(d_hi + offset) = pack_bf16x4(hx, hy, hz, hw);
    *reinterpret_cast<uint2*>(d_lo + offset) = pack_bf16x4(g.x - hx, g.y - hy, g.z - hz, g.w - hw);
  } else {
    st4(d_f32 + offset, g);
  }
}


// ---- the edge walks and the node epilogue, shared by the row kernels (tconv.cu) and the hub kernels (tconv_hub.cu)

// Edge metadata of one chunk of LPN edges of a lane group's row: lane `lig` of the group holds edge c0 + lig (`a` =
// col / row, `b` = eperm / cpos; `b` stays 0 when its array is NULL), loaded in one coalesced step.  The walks take an
// edge's indices from the lane that holds them (__shfl_sync), so the gathers of an unroll group wait on no index load;
// a row of more than LPN edges loads its further chunks as the walk reaches them.  The persistent kernels load chunk 0
// of a node's row while the previous node computes.
struct EdgeMeta { int32_t a, b; };
__device__ __forceinline__ EdgeMeta load_edge_meta(const int32_t* __restrict__ a, const int32_t* __restrict__ b,
                                                   int begin, int count, int c0, int lig) {
  EdgeMeta e{0, 0};
  if (c0 + lig < count) {
    e.a = a[begin + c0 + lig];
    if (b != nullptr) e.b = b[begin + c0 + lig];
  }
  return e;
}
// lane of this lane group that holds edge k of the current chunk
template <int DIM>
__device__ __forceinline__ int meta_lane(int k) { return ((threadIdx.x & 31) & ~(RowGeom<DIM>::LPN - 1)) + k; }

// Forward: one-pass online softmax over `count` in-edges starting at CSR position `begin` (count_max = the
// warp-uniform loop bound: the head reductions are warp shuffles).  m / l / acc are carried in and out.
// meta: chunk 0 of the row, load_edge_meta(col, alpha_mask ? eperm : NULL, begin, count, 0, lig).  The attention-mask
// value of an edge is loaded through its eperm together with the edge's key / value rows.
template <int DIM, int HEAD_DIM, int UNROLL>
__device__ __forceinline__ void fwd_edges(const float* __restrict__ qkvs, const float4 (&q)[RowGeom<DIM>::V],
                                          const int32_t* __restrict__ col, const int32_t* __restrict__ eperm,
                                          const float* __restrict__ alpha_mask, int begin, int count, int count_max,
                                          int64_t idle_row, int lig, EdgeMeta meta, float (&m)[RowGeom<DIM>::V],
                                          float (&l)[RowGeom<DIM>::V], float4 (&acc)[RowGeom<DIM>::V]) {
  constexpr int V = RowGeom<DIM>::V, LPN = RowGeom<DIM>::LPN;
  constexpr int HEADS = DIM / HEAD_DIM;
  static_assert(LPN % UNROLL == 0, "an unroll group must not straddle two metadata chunks");
  const float scale = rsqrtf((float)HEAD_DIM);
  for (int e0 = 0; e0 < count_max; e0 += UNROLL) {
    const int c0 = e0 & ~(LPN - 1);
    if (e0 == c0 && c0 > 0) meta = load_edge_meta(col, alpha_mask != nullptr ? eperm : nullptr, begin, count, c0, lig);
    float4 kr[UNROLL][V], vr[UNROLL][V];
    float mk[UNROLL][V];
    bool on[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      on[u] = e0 + u < count;
      const int j32 = __shfl_sync(0xffffffffu, meta.a, meta_lane<DIM>(e0 - c0 + u));
      const int64_t j = on[u] ? j32 : idle_row;
      const float* other = qkvs + j * 4 * DIM;
      load_row<DIM>(other + DIM, lig, kr[u]);
      load_row<DIM>(other + 2 * DIM, lig, vr[u]);
      if (alpha_mask != nullptr) {
        const int64_t ep = __shfl_sync(0xffffffffu, meta.b, meta_lane<DIM>(e0 - c0 + u));
#pragma unroll
        for (int v = 0; v < V; ++v) mk[u][v] = on[u] ? alpha_mask[ep * HEADS + head_of<DIM, HEAD_DIM>(v, lig)] : 0.f;
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      float a[V];
#pragma unroll
      for (int v = 0; v < V; ++v) a[v] = dot4(q[v], kr[u][v]);
      head_reduce<DIM, HEAD_DIM>(a);
      if (on[u]) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float logit = a[v] * scale;
          const float m_new = fmaxf(m[v], logit);
          const float corr = expf(m[v] - m_new);
          float p = expf(logit - m_new);
          l[v] = l[v] * corr + p;
          if (alpha_mask != nullptr) p *= mk[u][v];
          acc[v] = fma4(p, vr[u][v], scale4(corr, acc[v]));
          m[v] = m_new;
        }
      }
    }
  }
}

// Forward node epilogue, given the node's skip row xr: agg = acc / (l + eps), gate beta = sigmoid(w . [agg, x_r,
// agg - x_r]), out = beta x_r + (1 - beta) agg; saves agg, beta, m, 1/l.  Every lane of the warp must call it (group_sum shuffles); `store`
// says whether this lane group owns a row.
// `stats` (or NULL): this lane group's running column sums in shared memory, [sum o | sum o^2] as 2*DIM doubles (each
// lane owns its own slots): the BatchNorm statistics of the layer output, taken while the row is still in registers.
template <int DIM, int HEAD_DIM>
__device__ __forceinline__ void fwd_epilogue(const float4 (&xr)[RowGeom<DIM>::V], bool store, int64_t nrow, int lig,
                                             const float (&m)[RowGeom<DIM>::V], const float (&l)[RowGeom<DIM>::V],
                                             const float4 (&acc)[RowGeom<DIM>::V], const float* __restrict__ w_beta,
                                             float* __restrict__ out, float* __restrict__ agg_out,
                                             float* __restrict__ beta_out, float* __restrict__ m_out,
                                             float* __restrict__ invl_out, double* stats = nullptr) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  constexpr int HEADS = DIM / HEAD_DIM;
  constexpr int HEAD_F4 = HEAD_DIM / 4;
  float4 ag[V];
  float zpart = 0.f;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const float inv = 1.f / (l[v] + kSoftmaxEps);
    ag[v] = scale4(inv, acc[v]);
    const int f = v * LPN + lig;
    if (store && f % HEAD_F4 == 0) {
      m_out[nrow * HEADS + f / HEAD_F4] = m[v];
      invl_out[nrow * HEADS + f / HEAD_F4] = inv;
    }
    if (w_beta != nullptr) {
      const float4 w1 = ldg4(w_beta + 4 * f), w2 = ldg4(w_beta + DIM + 4 * f), w3 = ldg4(w_beta + 2 * DIM + 4 * f);
      zpart += dot4(w1, ag[v]) + dot4(w2, xr[v]) + dot4(w3, sub4(ag[v], xr[v]));
    }
  }
  float b = 0.f;
  if (w_beta != nullptr) {
    const float z = group_sum<LPN>(zpart);
    b = 1.f / (1.f + expf(-z));
  }
  if (!store) return;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int f = v * LPN + lig;
    float4 o;
    if (w_beta != nullptr) o = add4(scale4(b, xr[v]), scale4(1.f - b, ag[v]));
    else o = add4(ag[v], xr[v]);
    st4(out + nrow * DIM + 4 * f, o);
    st4(agg_out + nrow * DIM + 4 * f, ag[v]);
    if (stats != nullptr) {
      double* s0 = stats + 4 * f;
      double* s1 = stats + DIM + 4 * f;
      s0[0] += o.x; s0[1] += o.y; s0[2] += o.z; s0[3] += o.w;
      s1[0] += (double)o.x * o.x; s1[1] += (double)o.y * o.y; s1[2] += (double)o.z * o.z; s1[3] += (double)o.w * o.w;
    }
  }
  if (lig == 0 && beta_out != nullptr) beta_out[nrow] = b;
}

// Fixed-order reduction of the lane groups' column sums of one CTA into its partial row (the statistics variants of
// the forward kernels): every thread must call it.
template <int DIM>
__device__ __forceinline__ void stats_flush(const double* __restrict__ smem_stats, double* __restrict__ partial_row) {
  constexpr int NG = (kThreads / 32) * RowGeom<DIM>::GROUPS;
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * DIM; i += kThreads) {
    double s = 0.0;
    for (int g = 0; g < NG; ++g) s += smem_stats[(size_t)g * 2 * DIM + i];
    partial_row[i] = s;
  }
}

// Backward, destination side, one lane group per destination loading its edge indices as it goes: the dense-graph
// destination pass and the hub chunks, where the metadata-in-lanes walk below measured slower.  Over `count` in-edges of destination i starting at CSR position `begin`:
// alpha (recomputed from the saved m, 1/l), d_alpha = <d_agg_i, v_j>_h, d_logit = alpha (d_alpha mask - delta),
// dq += scale d_logit k_j; emits per-edge (alpha mask, scale d_logit) for the source pass.
template <int DIM, int HEAD_DIM, int UNROLL>
__device__ __forceinline__ void bwd_dst_edges_serial(const float* __restrict__ qkvs, const float4 (&q)[RowGeom<DIM>::V],
                                              const float4 (&dag)[RowGeom<DIM>::V],
                                              const float (&delta)[RowGeom<DIM>::V], const float (&mh)[RowGeom<DIM>::V],
                                              const float (&il)[RowGeom<DIM>::V], const int32_t* __restrict__ col,
                                              const int32_t* __restrict__ eperm, const float* __restrict__ alpha_mask,
                                              int begin, int count, int count_max, int64_t idle_row, int lig,
                                              float2* __restrict__ ecoef, float4 (&dq)[RowGeom<DIM>::V]) {
  constexpr int V = RowGeom<DIM>::V, LPN = RowGeom<DIM>::LPN;
  constexpr int HEADS = DIM / HEAD_DIM;
  constexpr int HEAD_F4 = HEAD_DIM / 4;
  const float scale = rsqrtf((float)HEAD_DIM);
  for (int e0 = 0; e0 < count_max; e0 += UNROLL) {
    float4 kr[UNROLL][V], vr[UNROLL][V];
    int pos[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const bool on = e0 + u < count;
      pos[u] = on ? begin + e0 + u : -1;
      const int64_t j = on ? col[pos[u]] : idle_row;
      const float* other = qkvs + j * 4 * DIM;
      load_row<DIM>(other + DIM, lig, kr[u]);
      load_row<DIM>(other + 2 * DIM, lig, vr[u]);
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      float a[V], da[V];
#pragma unroll
      for (int v = 0; v < V; ++v) { a[v] = dot4(q[v], kr[u][v]); da[v] = dot4(dag[v], vr[u][v]); }
      head_reduce<DIM, HEAD_DIM>(a);
      head_reduce<DIM, HEAD_DIM>(da);
      if (pos[u] >= 0) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float alpha = expf(a[v] * scale - mh[v]) * il[v];
          float mask = 1.f;
          const int h = head_of<DIM, HEAD_DIM>(v, lig);
          if (alpha_mask != nullptr) mask = alpha_mask[(int64_t)eperm[pos[u]] * HEADS + h];
          const float dlogit = alpha * (da[v] * mask - delta[v]) * scale;
          dq[v] = fma4(dlogit, kr[u][v], dq[v]);
          if ((v * LPN + lig) % HEAD_F4 == 0) ecoef[(int64_t)pos[u] * HEADS + h] = make_float2(alpha * mask, dlogit);
        }
      }
    }
  }
}

// Backward, destination side, session batches: over `count` in-edges of destination i starting at CSR position `begin`:
// alpha (recomputed from the saved m, 1/l), d_alpha = <d_agg_i, v_j>_h, d_logit = alpha (d_alpha mask - delta),
// dq += scale d_logit k_j; emits per-edge (alpha mask, scale d_logit) for the source pass.
// meta: chunk 0 of the row, as for fwd_edges.
template <int DIM, int HEAD_DIM, int UNROLL>
__device__ __forceinline__ void bwd_dst_edges(const float* __restrict__ qkvs, const float4 (&q)[RowGeom<DIM>::V],
                                              const float4 (&dag)[RowGeom<DIM>::V],
                                              const float (&delta)[RowGeom<DIM>::V], const float (&mh)[RowGeom<DIM>::V],
                                              const float (&il)[RowGeom<DIM>::V], const int32_t* __restrict__ col,
                                              const int32_t* __restrict__ eperm, const float* __restrict__ alpha_mask,
                                              int begin, int count, int count_max, int64_t idle_row, int lig,
                                              EdgeMeta meta, float2* __restrict__ ecoef, float4 (&dq)[RowGeom<DIM>::V]) {
  constexpr int V = RowGeom<DIM>::V, LPN = RowGeom<DIM>::LPN;
  constexpr int HEADS = DIM / HEAD_DIM;
  constexpr int HEAD_F4 = HEAD_DIM / 4;
  static_assert(LPN % UNROLL == 0, "an unroll group must not straddle two metadata chunks");
  const float scale = rsqrtf((float)HEAD_DIM);
  for (int c0 = 0; c0 < count_max; c0 += LPN) {
    if (c0 > 0) meta = load_edge_meta(col, alpha_mask != nullptr ? eperm : nullptr, begin, count, c0, lig);
    const int c_end = min(c0 + LPN, count_max);
    for (int e0 = c0; e0 < c_end; e0 += UNROLL) {
      float4 kr[UNROLL][V], vr[UNROLL][V];
      float mk[UNROLL][V];
      bool on[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        on[u] = e0 + u < count;
        const int j32 = __shfl_sync(0xffffffffu, meta.a, meta_lane<DIM>(e0 - c0 + u));
        const int64_t j = on[u] ? j32 : idle_row;
        const float* other = qkvs + j * 4 * DIM;
        load_row<DIM>(other + DIM, lig, kr[u]);
        load_row<DIM>(other + 2 * DIM, lig, vr[u]);
        if (alpha_mask != nullptr) {
          const int64_t ep = __shfl_sync(0xffffffffu, meta.b, meta_lane<DIM>(e0 - c0 + u));
#pragma unroll
          for (int v = 0; v < V; ++v) mk[u][v] = on[u] ? alpha_mask[ep * HEADS + head_of<DIM, HEAD_DIM>(v, lig)] : 0.f;
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        float a[V], da[V];
#pragma unroll
        for (int v = 0; v < V; ++v) { a[v] = dot4(q[v], kr[u][v]); da[v] = dot4(dag[v], vr[u][v]); }
        head_reduce<DIM, HEAD_DIM>(a);
        head_reduce<DIM, HEAD_DIM>(da);
        if (on[u]) {
#pragma unroll
          for (int v = 0; v < V; ++v) {
            const float alpha = expf(a[v] * scale - mh[v]) * il[v];
            const float mask = alpha_mask != nullptr ? mk[u][v] : 1.f;
            const int h = head_of<DIM, HEAD_DIM>(v, lig);
            const float dlogit = alpha * (da[v] * mask - delta[v]) * scale;
            dq[v] = fma4(dlogit, kr[u][v], dq[v]);
            if ((v * LPN + lig) % HEAD_F4 == 0)
              ecoef[(int64_t)(begin + e0 + u) * HEADS + h] = make_float2(alpha * mask, dlogit);
          }
        }
      }
    }
  }
}

// Backward, source side, one lane group per source walking its own edges (no shuffles, no warp-uniform bound): the
// dense-graph source pass and the hub chunks, where the metadata-in-lanes walk below measured slower (on dense rows
// its registers cost a resident CTA).  Over CSC positions [p0, p1) of source j: dk += scale d_logit_e q_i,
// dv += alpha_e mask_e d_agg_i (coefficients written by the destination pass in CSR order, found through cpos).
template <int DIM, int HEAD_DIM>
__device__ __forceinline__ void bwd_src_edges_serial(const float* __restrict__ qkvs, const float* __restrict__ d_agg,
                                                     const float2* __restrict__ ecoef, const int32_t* __restrict__ row,
                                                     const int32_t* __restrict__ cpos, int p_begin, int p_end, int lig,
                                                     float4 (&dk)[RowGeom<DIM>::V], float4 (&dv)[RowGeom<DIM>::V]) {
  constexpr int V = RowGeom<DIM>::V;
  constexpr int HEADS = DIM / HEAD_DIM;
  for (int p0 = p_begin; p0 < p_end; p0 += kEdgeUnroll) {
    float4 qr[kEdgeUnroll][V], gr[kEdgeUnroll][V];
    float2 c[kEdgeUnroll][V];
#pragma unroll
    for (int u = 0; u < kEdgeUnroll; ++u) {
      const bool on = p0 + u < p_end;
      const int p = on ? p0 + u : p_begin;
      const int64_t i = row[p];
      const int64_t e = cpos[p];
      load_row<DIM>(qkvs + i * 4 * DIM, lig, qr[u]);
      load_row<DIM>(d_agg + i * DIM, lig, gr[u]);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        c[u][v] = ecoef[e * HEADS + head_of<DIM, HEAD_DIM>(v, lig)];
        if (!on) c[u][v] = make_float2(0.f, 0.f);
      }
    }
#pragma unroll
    for (int u = 0; u < kEdgeUnroll; ++u) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        dk[v] = fma4(c[u][v].y, qr[u][v], dk[v]);
        dv[v] = fma4(c[u][v].x, gr[u][v], dv[v]);
      }
    }
  }
}

// Backward, source side, session batches: over the `count` CSC positions from p_begin of source j (count_max = the warp-uniform loop
// bound): dk += scale d_logit_e q_i, dv += alpha_e mask_e d_agg_i (coefficients written by the destination pass in
// CSR order, found through cpos).  meta: chunk 0, load_edge_meta(row, cpos, p_begin, count, 0, lig); an edge's
// coefficients are loaded with its q and d_agg rows.
template <int DIM, int HEAD_DIM, int UNROLL>
__device__ __forceinline__ void bwd_src_edges(const float* __restrict__ qkvs, const float* __restrict__ d_agg,
                                              const float2* __restrict__ ecoef, const int32_t* __restrict__ row,
                                              const int32_t* __restrict__ cpos, int p_begin, int count, int count_max,
                                              int lig, EdgeMeta meta, float4 (&dk)[RowGeom<DIM>::V],
                                              float4 (&dv)[RowGeom<DIM>::V]) {
  constexpr int V = RowGeom<DIM>::V, LPN = RowGeom<DIM>::LPN;
  constexpr int HEADS = DIM / HEAD_DIM;
  static_assert(LPN % UNROLL == 0, "an unroll group must not straddle two metadata chunks");
  for (int c0 = 0; c0 < count_max; c0 += LPN) {
    if (c0 > 0) meta = load_edge_meta(row, cpos, p_begin, count, c0, lig);
    const int c_end = min(c0 + LPN, count_max);
    for (int e0 = c0; e0 < c_end; e0 += UNROLL) {
      float4 qr[UNROLL][V], gr[UNROLL][V];
      float2 c[UNROLL][V];
      bool on[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        // an edge past the row's end reads row 0 and edge 0 (a lane past its node's edges holds zeros) and adds
        // nothing: its coefficients are zero
        on[u] = e0 + u < count;
        const int64_t i = __shfl_sync(0xffffffffu, meta.a, meta_lane<DIM>(e0 - c0 + u));
        const int64_t e = __shfl_sync(0xffffffffu, meta.b, meta_lane<DIM>(e0 - c0 + u));
        load_row<DIM>(qkvs + i * 4 * DIM, lig, qr[u]);
        load_row<DIM>(d_agg + i * DIM, lig, gr[u]);
#pragma unroll
        for (int v = 0; v < V; ++v) {
          c[u][v] = ecoef[e * HEADS + head_of<DIM, HEAD_DIM>(v, lig)];
          if (!on[u]) c[u][v] = make_float2(0.f, 0.f);
        }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          dk[v] = fma4(c[u][v].y, qr[u][v], dk[v]);
          dv[v] = fma4(c[u][v].x, gr[u][v], dv[v]);
        }
      }
    }
  }
}

}  // namespace

// ---- hub rows ---------------------------------------------------------------------------------------------------
// A destination (or, in the backward source pass, a source) with more than kHubThreshold edges is a *hub*: one lane
// group walking its edges serially would take milliseconds on a power-law graph (the reference's own generator is
// zipf(1.5), scripts/data/00_generate_synthetic_data.py:53; the 1M-item graph has rows of 80,000 edges).  Hub rows are
// cut into chunks of kHubChunk edges; a CTA processes one chunk with the row's query (and d_agg) staged in shared
// memory, its lane groups each take a slice, and their (m, l, acc) / gradient partials are combined in a fixed order —
// first inside the CTA, then over the chunks of the row.  The plan (which rows, which chunks) is built once per graph
// index by etpgt_hub_plan, deterministically (prefix sums, no atomics).
constexpr int kHubThreshold = 256;
constexpr int kHubChunk = 256;

struct HubRow { int32_t node, first_chunk, num_chunks, pad; };
struct HubChunk { int32_t node, edge_begin, edge_count, slot; };

// Layout of the plan buffer (int32 units), identical for the CSR (destination) and CSC (source) halves.
struct HubPlanView {
  int32_t* counts;       // [4]: dst hubs, dst chunks, src hubs, src chunks
  HubRow* dst_rows;      // [cap_rows]
  HubChunk* dst_chunks;  // [cap_chunks]
  HubRow* src_rows;
  HubChunk* src_chunks;
  int64_t cap_rows, cap_chunks;
};
inline int64_t hub_cap_rows(int64_t num_edges) { return num_edges / (kHubThreshold + 1) + 1; }
inline int64_t hub_cap_chunks(int64_t num_edges) { return num_edges / kHubChunk + hub_cap_rows(num_edges) + 1; }
inline size_t hub_plan_bytes(int64_t num_edges) {
  return 256 + 2 * (align_up((size_t)hub_cap_rows(num_edges) * sizeof(HubRow)) +
                    align_up((size_t)hub_cap_chunks(num_edges) * sizeof(HubChunk)));
}
inline HubPlanView hub_plan_view(void* plan, int64_t num_edges) {
  HubPlanView v;
  char* p = static_cast<char*>(plan);
  v.cap_rows = hub_cap_rows(num_edges);
  v.cap_chunks = hub_cap_chunks(num_edges);
  v.counts = reinterpret_cast<int32_t*>(p);
  p += 256;
  v.dst_rows = reinterpret_cast<HubRow*>(p);
  p += align_up((size_t)v.cap_rows * sizeof(HubRow));
  v.dst_chunks = reinterpret_cast<HubChunk*>(p);
  p += align_up((size_t)v.cap_chunks * sizeof(HubChunk));
  v.src_rows = reinterpret_cast<HubRow*>(p);
  p += align_up((size_t)v.cap_rows * sizeof(HubRow));
  v.src_chunks = reinterpret_cast<HubChunk*>(p);
  return v;
}

// tconv_hub.cu: the hub halves of the three passes (launched by tconv.cu after its own row kernels, which skip rows
// with more than kHubThreshold edges when a plan is given).  `hub_ws` holds the per-chunk partials.
constexpr int kHubColsumCtas = 32;   // CTAs (= partial rows) of the hub combine kernels: 256 rows in one round at dim 256
// stat_rows (or NULL): kHubColsumCtas rows of 2*dim doubles receiving the hub rows' [sum out | sum out^2]
int tconv_fwd_hubs(const float* qkvs, int dim, int heads, const int32_t* col, const int32_t* eperm,
                   int64_t num_edges, const float* w_beta, const float* alpha_mask, float* out, float* agg, float* beta,
                   float* m, float* inv_l, const void* hub_plan, void* hub_ws, double* stat_rows, cudaStream_t stream);
// dq of hub destinations; colsum_rows (or NULL): kHubColsumCtas rows of `width` floats whose columns
// [col_offset, col_offset + dim) receive the column sums of those dq rows (the other columns are zeroed)
int tconv_bwd_dst_hubs(const float* qkvs, int dim, int heads, const int32_t* col, const int32_t* eperm,
                       int64_t num_edges, const float* alpha_mask, const float* agg, const float* m, const float* inv_l,
                       const float* d_agg, float2* ecoef, float* d_qkvs, __nv_bfloat16* d_hi, __nv_bfloat16* d_lo,
                       float* colsum_rows, int width, int col_offset, const void* hub_plan, void* hub_ws,
                       cudaStream_t stream);
// dk, dv of hub sources; colsum_rows (or NULL): kHubColsumCtas rows of 2*dim floats (key | value column sums)
int tconv_bwd_src_hubs(const float* qkvs, int dim, int heads, const int32_t* row, const int32_t* cpos,
                       int64_t num_edges, const float* d_agg, const float2* ecoef, float* d_qkvs, __nv_bfloat16* d_hi,
                       __nv_bfloat16* d_lo, float* colsum_rows, const void* hub_plan, void* hub_ws, cudaStream_t stream);

}  // namespace etpgt
