// a12: GAT edge-softmax + aggregation (PyG GATConv, add_self_loops=True) and GraphSAGE mean
// aggregation over the same CSR / CSC index.  etpgt/model/gat.py:49-109,137;
// etpgt/model/graphsage.py:43-48,75 (semantics: SURVEY.md Appendix A, oracle/conv_ref.py).
//
// GAT: h [N, W] with W = heads*C is the projected feature row (one GEMM by the caller) and
// a_src / a_dst [N, heads] the per-head attention scalars.  Logits are scalars per (edge,
// head), so the only gathered data is h_j.  Existing self loops are skipped and exactly one
// self loop per node is processed after the real edges (PyG remove_self_loops +
// add_self_loops).  Gather-bound: W*4 B per edge + 2*W*4 B per node forward.
#include <math.h>

#include <cuda_bf16.h>

#include "common.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;
constexpr float kSoftmaxEps = 1e-16f;

template <int W>
struct GatGeom : RowGeom<W> {
  static constexpr int UNROLL = RowGeom<W>::V >= 8 ? 2 : 4;
};

template <int W>
__device__ __forceinline__ void load_row(const float* __restrict__ row, int lig, float4 (&dst)[RowGeom<W>::V]) {
#pragma unroll
  for (int v = 0; v < RowGeom<W>::V; ++v) dst[v] = ldg4(row + 4 * (v * RowGeom<W>::LPN + lig));
}
// the gradient row of the per-head result when only d(head mean) [N, C] exists: d_agg[n, h, c] = d_out[n, c] / H
template <int W, int C>
__device__ __forceinline__ void load_grad_row(const float* __restrict__ d_agg, const float* __restrict__ d_out_mean,
                                              int64_t node, int lig, float4 (&dst)[RowGeom<W>::V]) {
  if (d_out_mean == nullptr) {
    load_row<W>(d_agg + node * W, lig, dst);
    return;
  }
  constexpr int HEAD_F4 = C / 4;
  const float inv = 1.f / (float)(W / C);
#pragma unroll
  for (int v = 0; v < RowGeom<W>::V; ++v)
    dst[v] = scale4(inv, ldg4(d_out_mean + node * C + 4 * ((v * RowGeom<W>::LPN + lig) % HEAD_F4)));
}

__device__ __forceinline__ float leaky(float z, float slope) { return z > 0.f ? z : slope * z; }

// --------------------------------------------------------------------------- GAT forward
template <int W, int C>
__global__ void __launch_bounds__(kThreads, 2)
gat_fwd_kernel(const float* __restrict__ h, const float* __restrict__ a_src, const float* __restrict__ a_dst,
               int64_t num_nodes, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
               const int32_t* __restrict__ eperm, float slope, const float* __restrict__ mask_edges,
               const float* __restrict__ mask_self, float* __restrict__ agg, float* __restrict__ m_out,
               float* __restrict__ invl_out, const float* __restrict__ bias, float* __restrict__ out_mean) {
  using G = GatGeom<W>;
  constexpr int V = G::V, LPN = G::LPN, HEADS = W / C, HEAD_F4 = C / 4, U = G::UNROLL;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t node = ((blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5) * G::GROUPS + lane / LPN;
  if (node >= num_nodes) return;  // no warp collectives in the forward
  int hd[V];
  float ad[V], m[V], l[V];
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) {
    hd[v] = head_of<W, C>(v, lig);
    ad[v] = a_dst[node * HEADS + hd[v]];
    m[v] = -INFINITY; l[v] = 0.f; acc[v] = zero4();
  }
  const int begin = rowptr[node], end = rowptr[node + 1];
  // the appended self loop is folded in as one extra trip (p == end)
  for (int p0 = begin; p0 <= end; p0 += U) {
    float4 hr[U][V];
    int64_t src[U];
    int pp[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = p0 + u;
      pp[u] = p;
      src[u] = p < end ? col[p] : node;
      load_row<W>(h + src[u] * W, lig, hr[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = pp[u];
      const bool is_self = p == end;
      if (p > end || (!is_self && src[u] == node)) continue;  // beyond the row, or a dropped self loop
      if constexpr (HEAD_F4 % LPN == 0) {
        // a head covers whole slots (the reference's width: 2 slots per head): logit, running max / sum and the two
        // exponentials once per HEAD instead of once per slot
        constexpr int VH = HEAD_F4 / LPN;
#pragma unroll
        for (int hh = 0; hh < HEADS; ++hh) {
          const int v0 = hh * VH;
          const float logit = leaky(a_src[src[u] * HEADS + hh] + ad[v0], slope);
          const float m_new = fmaxf(m[v0], logit);
          const float corr = expf(m[v0] - m_new);
          float pr = expf(logit - m_new);
          const float l_new = l[v0] * corr + pr;
          if (mask_edges != nullptr)
            pr *= is_self ? mask_self[node * HEADS + hh] : mask_edges[(int64_t)eperm[p] * HEADS + hh];
#pragma unroll
          for (int vv = 0; vv < VH; ++vv) {
            acc[v0 + vv] = fma4(pr, hr[u][v0 + vv], scale4(corr, acc[v0 + vv]));
            m[v0 + vv] = m_new;
            l[v0 + vv] = l_new;
          }
        }
      } else {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          const float logit = leaky(a_src[src[u] * HEADS + hd[v]] + ad[v], slope);
          const float m_new = fmaxf(m[v], logit);
          const float corr = expf(m[v] - m_new);
          float pr = expf(logit - m_new);
          l[v] = l[v] * corr + pr;
          if (mask_edges != nullptr)
            pr *= is_self ? mask_self[node * HEADS + hd[v]] : mask_edges[(int64_t)eperm[p] * HEADS + hd[v]];
          acc[v] = fma4(pr, hr[u][v], scale4(corr, acc[v]));
          m[v] = m_new;
        }
      }
    }
  }
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const float inv = 1.f / (l[v] + kSoftmaxEps);
    const int f = v * LPN + lig;
    acc[v] = scale4(inv, acc[v]);
    st4(agg + node * W + 4 * f, acc[v]);
    if (f % HEAD_F4 == 0) { m_out[node * HEADS + hd[v]] = m[v]; invl_out[node * HEADS + hd[v]] = inv; }
  }
  // concat=False (etpgt/model/gat.py:100-109): mean over the heads + bias, written next to the per-head rows (kept
  // for the backward pass).  When a head spans whole lane-group rounds (C/4 a multiple of the lanes per node) the
  // H values of an output column sit in the same lane: no shuffles, no second pass over [N, heads*C].
  if constexpr (HEAD_F4 % LPN == 0) {
    if (out_mean != nullptr) {
      constexpr int VH = HEAD_F4 / LPN;   // float4 slots per head and lane
#pragma unroll
      for (int vv = 0; vv < VH; ++vv) {
        float4 s = acc[vv];
#pragma unroll
        for (int hh = 1; hh < HEADS; ++hh) s = add4(s, acc[hh * VH + vv]);   // head order 0..H-1, as the separate pass
        s = scale4(1.f / (float)HEADS, s);
        const int f = vv * LPN + lig;
        if (bias != nullptr) s = add4(s, ldg4(bias + 4 * f));
        st4(out_mean + node * C + 4 * f, s);
      }
    }
  }
}

// ------------------------------------------------------------- GAT backward, destination pass
// delta_h = <d_agg_i, agg_i>_h; per edge: alpha from saved (m, 1/l), d_alpha = <d_agg_i, h_j>_h,
// d_e = alpha (d_alpha*mask - delta), d_z = d_e * leaky'(z).  Writes d_a_dst[i,h] = sum d_z and the
// per-edge / per-self-loop coefficients (alpha*mask, d_z) for the source pass.
template <int W, int C>
__global__ void __launch_bounds__(kThreads, 2)
gat_bwd_dst_kernel(const float* __restrict__ h, const float* __restrict__ a_src, const float* __restrict__ a_dst,
                   const float* __restrict__ d_agg, const float* __restrict__ agg, int64_t num_nodes,
                   const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                   const int32_t* __restrict__ eperm, float slope, const float* __restrict__ mask_edges,
                   const float* __restrict__ mask_self, const float* __restrict__ m_in,
                   const float* __restrict__ invl_in, float2* __restrict__ ecoef, float2* __restrict__ self_coef,
                   float* __restrict__ d_a_dst, const float* __restrict__ d_out_mean) {
  using G = GatGeom<W>;
  constexpr int V = G::V, LPN = G::LPN, HEADS = W / C, HEAD_F4 = C / 4, U = G::UNROLL;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t warp_base = ((blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5) * G::GROUPS;
  if (warp_base >= num_nodes) return;  // warp-uniform
  const int64_t node = warp_base + lane / LPN;
  const bool valid = node < num_nodes;
  const int64_t nrow = valid ? node : 0;

  int hd[V];
  float ad[V], mh[V], il[V], delta[V], dsum[V];
  float4 g[V];
  {
    float4 ag[V];
    load_grad_row<W, C>(d_agg, d_out_mean, nrow, lig, g);
    load_row<W>(agg + nrow * W, lig, ag);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      hd[v] = head_of<W, C>(v, lig);
      ad[v] = a_dst[nrow * HEADS + hd[v]];
      mh[v] = m_in[nrow * HEADS + hd[v]];
      il[v] = invl_in[nrow * HEADS + hd[v]];
      delta[v] = dot4(g[v], ag[v]);
      dsum[v] = 0.f;
    }
  }
  head_reduce<W, C>(delta);
  const int begin = valid ? rowptr[nrow] : 0;
  const int end = valid ? rowptr[nrow + 1] : -1;  // invalid groups take zero trips (end - begin + 1 = 0)
  int trips = end - begin + 1, trips_max = trips;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) trips_max = max(trips_max, __shfl_xor_sync(0xffffffffu, trips_max, off));

  for (int t0 = 0; t0 < trips_max; t0 += U) {
    float4 hr[U][V];
    int64_t src[U];
    int pp[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = begin + t0 + u;
      pp[u] = p;
      src[u] = (valid && p < end) ? col[p] : nrow;
      load_row<W>(h + src[u] * W, lig, hr[u]);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int p = pp[u];
      const bool is_self = p == end;
      const bool on = valid && p <= end;
      const bool dropped = on && !is_self && src[u] == nrow;
      if constexpr (HEAD_F4 % LPN == 0) {
        // a head covers whole slots: ONE butterfly per head over the sum of its slots (20 instead of 40 shuffles per
        // edge at four heads), alpha / leaky' / masks once per head
        constexpr int VH = HEAD_F4 / LPN;
        float dah[HEADS];
#pragma unroll
        for (int hh = 0; hh < HEADS; ++hh) {
          float sacc = 0.f;
#pragma unroll
          for (int vv = 0; vv < VH; ++vv) sacc += dot4(g[hh * VH + vv], hr[u][hh * VH + vv]);
          dah[hh] = group_sum<LPN>(sacc);
        }
        if (on) {
#pragma unroll
          for (int hh = 0; hh < HEADS; ++hh) {
            const int v0 = hh * VH;
            float2 c = make_float2(0.f, 0.f);
            if (!dropped) {
              const float z = a_src[src[u] * HEADS + hh] + ad[v0];
              const float alpha = expf(leaky(z, slope) - mh[v0]) * il[v0];
              float mask = 1.f;
              if (mask_edges != nullptr)
                mask = is_self ? mask_self[nrow * HEADS + hh] : mask_edges[(int64_t)eperm[p] * HEADS + hh];
              const float dz = alpha * (dah[hh] * mask - delta[v0]) * (z > 0.f ? 1.f : slope);
#pragma unroll
              for (int vv = 0; vv < VH; ++vv) dsum[v0 + vv] += dz;
              c = make_float2(alpha * mask, dz);
            }
            if (lig == 0) {
              if (is_self) self_coef[nrow * HEADS + hh] = c;
              else ecoef[(int64_t)p * HEADS + hh] = c;
            }
          }
        }
        continue;
      }
      float da[V];
#pragma unroll
      for (int v = 0; v < V; ++v) da[v] = dot4(g[v], hr[u][v]);
      head_reduce<W, C>(da);
      if (on) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
          float2 c = make_float2(0.f, 0.f);
          if (!dropped) {
            const float z = a_src[src[u] * HEADS + hd[v]] + ad[v];
            const float alpha = expf(leaky(z, slope) - mh[v]) * il[v];
            float mask = 1.f;
            if (mask_edges != nullptr)
              mask = is_self ? mask_self[nrow * HEADS + hd[v]] : mask_edges[(int64_t)eperm[p] * HEADS + hd[v]];
            const float dz = alpha * (da[v] * mask - delta[v]) * (z > 0.f ? 1.f : slope);
            dsum[v] += dz;
            c = make_float2(alpha * mask, dz);
          }
          if ((v * LPN + lig) % HEAD_F4 == 0) {
            if (is_self) self_coef[nrow * HEADS + hd[v]] = c;
            else ecoef[(int64_t)p * HEADS + hd[v]] = c;
          }
        }
      }
    }
  }
  if (valid) {
#pragma unroll
    for (int v = 0; v < V; ++v)
      if ((v * LPN + lig) % HEAD_F4 == 0) d_a_dst[nrow * HEADS + hd[v]] = dsum[v];
  }
}

// ------------------------------------------------------------------ GAT backward, source pass
template <int W, int C>
__global__ void __launch_bounds__(kThreads)
gat_bwd_src_kernel(const float* __restrict__ d_agg, int64_t num_nodes, const int32_t* __restrict__ colptr,
                   const int32_t* __restrict__ row, const int32_t* __restrict__ cpos,
                   const float2* __restrict__ ecoef, const float2* __restrict__ self_coef,
                   float* __restrict__ d_h, float* __restrict__ d_a_src, const float* __restrict__ d_out_mean,
                   __nv_bfloat16* __restrict__ d_h_hi, __nv_bfloat16* __restrict__ d_h_lo) {
  using G = GatGeom<W>;
  constexpr int V = G::V, LPN = G::LPN, HEADS = W / C, HEAD_F4 = C / 4;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t node = ((blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5) * G::GROUPS + lane / LPN;
  if (node >= num_nodes) return;
  int hd[V];
  float dsum[V];
  float4 acc[V], g[V];
  load_grad_row<W, C>(d_agg, d_out_mean, node, lig, g);
#pragma unroll
  for (int v = 0; v < V; ++v) {
    hd[v] = head_of<W, C>(v, lig);
    const float2 c = self_coef[node * HEADS + hd[v]];
    acc[v] = scale4(c.x, g[v]);
    dsum[v] = c.y;
  }
  const int begin = colptr[node], end = colptr[node + 1];
  for (int p = begin; p < end; ++p) {
    const int64_t i = row[p];
    const int64_t e = cpos[p];
    load_grad_row<W, C>(d_agg, d_out_mean, i, lig, g);   // [N, C]: a quarter of the gathered bytes at four heads
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const float2 c = ecoef[e * HEADS + hd[v]];  // (0,0) for dropped self loops
      acc[v] = fma4(c.x, g[v], acc[v]);
      dsum[v] += c.y;
    }
  }
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const int f = v * LPN + lig;
    if (d_h_hi != nullptr) {   // straight to the split-bf16 operands of the two projection-gradient GEMMs
      const float e[4] = {acc[v].x, acc[v].y, acc[v].z, acc[v].w};
      uint32_t hw[2], lw[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const __nv_bfloat16 h0 = __float2bfloat16_rn(e[2 * t]), h1 = __float2bfloat16_rn(e[2 * t + 1]);
        const __nv_bfloat16 l0 = __float2bfloat16_rn(e[2 * t] - __bfloat162float(h0));
        const __nv_bfloat16 l1 = __float2bfloat16_rn(e[2 * t + 1] - __bfloat162float(h1));
        hw[t] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        lw[t] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      }
      *reinterpret_cast<uint2*>(d_h_hi + node * W + 4 * f) = make_uint2(hw[0], hw[1]);
      *reinterpret_cast<uint2*>(d_h_lo + node * W + 4 * f) = make_uint2(lw[0], lw[1]);
    } else {
      st4(d_h + node * W + 4 * f, acc[v]);
    }
    if (f % HEAD_F4 == 0) d_a_src[node * HEADS + hd[v]] = dsum[v];
  }
}

// ------------------------------------------------------------------------- GraphSAGE mean
template <int DIM>
__global__ void __launch_bounds__(kThreads)
sage_mean_fwd_kernel(const float* __restrict__ x, int64_t num_nodes, const int32_t* __restrict__ rowptr,
                     const int32_t* __restrict__ col, float* __restrict__ mean, __nv_bfloat16* __restrict__ mean_hi,
                     __nv_bfloat16* __restrict__ mean_lo, int64_t ld) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t node = ((blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5) * G::GROUPS + lane / LPN;
  if (node >= num_nodes) return;
  const int begin = rowptr[node], end = rowptr[node + 1];
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = zero4();
  for (int p0 = begin; p0 < end; p0 += 4) {
    float4 r[4][V];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t j = p0 + u < end ? col[p0 + u] : node;
      load_row<DIM>(x + j * DIM, lig, r[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (p0 + u < end)
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] = add4(acc[v], r[u][v]);
  }
  const float inv = end > begin ? 1.f / (float)(end - begin) : 0.f;
#pragma unroll
  for (int v = 0; v < V; ++v) {
    const float4 r = scale4(inv, acc[v]);
    if (mean != nullptr) st4(mean + node * DIM + 4 * (v * LPN + lig), r);
    if (mean_hi != nullptr) {   // straight into (a column block of) the split-bf16 operand of the layer's GEMM
      const float e[4] = {r.x, r.y, r.z, r.w};
      uint32_t hw[2], lw[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        const __nv_bfloat16 h0 = __float2bfloat16_rn(e[2 * t]), h1 = __float2bfloat16_rn(e[2 * t + 1]);
        const __nv_bfloat16 l0 = __float2bfloat16_rn(e[2 * t] - __bfloat162float(h0));
        const __nv_bfloat16 l1 = __float2bfloat16_rn(e[2 * t + 1] - __bfloat162float(h1));
        hw[t] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        lw[t] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      }
      *reinterpret_cast<uint2*>(mean_hi + node * ld + 4 * (v * LPN + lig)) = make_uint2(hw[0], hw[1]);
      *reinterpret_cast<uint2*>(mean_lo + node * ld + 4 * (v * LPN + lig)) = make_uint2(lw[0], lw[1]);
    }
  }
}

// d_x_j = sum over out-edges (j -> i) of d_mean_i / indeg(i)  (+ d_root_j: the lin_r branch of SAGEConv, when the two
// gradients arrive as the column halves of one [N, 2*DIM] GEMM output — `ld` is that pitch)
template <int DIM>
__global__ void __launch_bounds__(kThreads)
sage_mean_bwd_kernel(const float* __restrict__ d_mean, int64_t ld, const float* __restrict__ d_root,
                     int64_t num_nodes, const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colptr,
                     const int32_t* __restrict__ row, float* __restrict__ d_x) {
  using G = RowGeom<DIM>;
  constexpr int V = G::V, LPN = G::LPN;
  const int lane = threadIdx.x & 31;
  const int lig = lane % LPN;
  const int64_t node = ((blockIdx.x * (int64_t)kThreads + threadIdx.x) >> 5) * G::GROUPS + lane / LPN;
  if (node >= num_nodes) return;
  float4 acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v)
    acc[v] = d_root != nullptr ? ldg4(d_root + node * ld + 4 * (v * LPN + lig)) : zero4();
  for (int p = colptr[node]; p < colptr[node + 1]; ++p) {
    const int64_t i = row[p];
    const float inv = 1.f / (float)(rowptr[i + 1] - rowptr[i]);
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = fma4(inv, ldg4(d_mean + i * ld + 4 * (v * LPN + lig)), acc[v]);
  }
#pragma unroll
  for (int v = 0; v < V; ++v) st4(d_x + node * DIM + 4 * (v * LPN + lig), acc[v]);
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

#define ETPGT_GAT_CASE(W_, H_, CALL) \
  case (W_) * 16 + (H_): { CALL(W_, ((W_) / (H_))); } break;
#define ETPGT_GAT_ROW(W_, CALL) \
  ETPGT_GAT_CASE(W_, 1, CALL) ETPGT_GAT_CASE(W_, 2, CALL) ETPGT_GAT_CASE(W_, 4, CALL) ETPGT_GAT_CASE(W_, 8, CALL)
#define ETPGT_DISPATCH_GAT(width, heads, CALL)                                                      \
  switch ((width) * 16 + (heads)) {                                                                 \
    ETPGT_GAT_ROW(32, CALL) ETPGT_GAT_ROW(64, CALL) ETPGT_GAT_ROW(128, CALL) ETPGT_GAT_ROW(256, CALL) \
    ETPGT_GAT_ROW(512, CALL) ETPGT_GAT_ROW(1024, CALL)                                              \
    default:                                                                                        \
      set_error("gat: unsupported (heads*channels=%d, heads=%d): width in {32..1024} powers of two, " \
                "heads in {1,2,4,8}", (int)(width), (int)(heads));                                  \
      return ETPGT_EINVAL;                                                                          \
  }

extern "C" int etpgt_gat_mean_fused_supported(int width, int heads) {
  if (heads < 1 || width % heads != 0) return 0;
  const int lpn = width / 4 < 32 ? width / 4 : 32;
  return lpn > 0 && (width / heads / 4) % lpn == 0 ? 1 : 0;
}

extern "C" int etpgt_gat_fwd_mean(const float* h, const float* a_src, const float* a_dst, int64_t num_nodes, int width,
                                  int heads, const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                                  float negative_slope, const float* mask_edges, const float* mask_self,
                                  const float* bias, float* agg, float* m, float* inv_l, float* out_mean,
                                  etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_nodes >= 0 && h && a_src && a_dst && rowptr && agg && m && inv_l, "gat_fwd: bad arguments");
  ETPGT_REQUIRE((mask_edges == nullptr) == (mask_self == nullptr), "gat_fwd: pass both masks or neither");
  ETPGT_REQUIRE(out_mean == nullptr || etpgt_gat_mean_fused_supported(width, heads),
                "gat_fwd_mean: the fused head mean needs channels/4 to be a multiple of the lanes per node "
                "(width=%d heads=%d)", width, heads);
  if (num_nodes == 0) return ETPGT_OK;
#define CALL(W, C)                                                                                        \
  {                                                                                                       \
    const int64_t npc = (kThreads / 32) * RowGeom<W>::GROUPS;                                             \
    gat_fwd_kernel<W, C><<<(unsigned)((num_nodes + npc - 1) / npc), kThreads, 0, stream>>>(                \
        h, a_src, a_dst, num_nodes, rowptr, col, eperm, negative_slope, mask_edges, mask_self, agg, m, inv_l, bias, \
        out_mean);                                                                                        \
  }
  ETPGT_DISPATCH_GAT(width, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("gat_fwd");
  return ETPGT_OK;
}

extern "C" int etpgt_gat_fwd(const float* h, const float* a_src, const float* a_dst, int64_t num_nodes, int width,
                             int heads, const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                             float negative_slope, const float* mask_edges, const float* mask_self, float* agg,
                             float* m, float* inv_l, etpgt_stream_t stream) {
  return etpgt_gat_fwd_mean(h, a_src, a_dst, num_nodes, width, heads, rowptr, col, eperm, negative_slope, mask_edges,
                            mask_self, nullptr, agg, m, inv_l, nullptr, stream);
}

extern "C" size_t etpgt_gat_bwd_workspace_bytes(int64_t num_nodes, int64_t num_edges, int heads) {
  return align_up((size_t)(num_edges > 0 ? num_edges : 1) * heads * sizeof(float2)) +
         align_up((size_t)(num_nodes > 0 ? num_nodes : 1) * heads * sizeof(float2)) + 256;
}

extern "C" int etpgt_gat_bwd_mean(const float* h, const float* a_src, const float* a_dst, const float* d_agg,
                                  const float* d_out_mean, const float* agg, int64_t num_nodes, int width, int heads,
                                  const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                                  const int32_t* colptr, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                                  float negative_slope, const float* mask_edges, const float* mask_self,
                                  const float* m, const float* inv_l, float* d_h, void* d_h_hi, void* d_h_lo,
                                  float* d_a_src, float* d_a_dst, void* ws, size_t ws_bytes,
                                  etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(num_nodes >= 0 && num_edges >= 0 && h && a_src && a_dst && agg && rowptr && colptr && m &&
                    inv_l && d_a_src && d_a_dst && (d_agg != nullptr) != (d_out_mean != nullptr),
                "gat_bwd: bad arguments (exactly one of d_agg [N, heads*C] and d_out_mean [N, C])");
  ETPGT_REQUIRE((d_h != nullptr) != (d_h_hi != nullptr) && (d_h_hi == nullptr) == (d_h_lo == nullptr),
                "gat_bwd: the projection gradient goes EITHER to d_h (fp32) or to d_h_hi / d_h_lo (split bf16)");
  ETPGT_REQUIRE((mask_edges == nullptr) == (mask_self == nullptr), "gat_bwd: pass both masks or neither");
  if (ws_bytes < etpgt_gat_bwd_workspace_bytes(num_nodes, num_edges, heads)) {
    set_error("gat_bwd: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  if (num_nodes == 0) return ETPGT_OK;
  Workspace w(ws, ws_bytes);
  float2* ecoef = w.take<float2>((size_t)(num_edges > 0 ? num_edges : 1) * heads);
  float2* self_coef = w.take<float2>((size_t)num_nodes * heads);
#define CALL(W, C)                                                                                          \
  {                                                                                                         \
    const int64_t npc = (kThreads / 32) * RowGeom<W>::GROUPS;                                               \
    const unsigned grid = (unsigned)((num_nodes + npc - 1) / npc);                                          \
    gat_bwd_dst_kernel<W, C><<<grid, kThreads, 0, stream>>>(h, a_src, a_dst, d_agg, agg, num_nodes, rowptr, col, eperm, \
                                                           negative_slope, mask_edges, mask_self, m, inv_l, ecoef, \
                                                           self_coef, d_a_dst, d_out_mean);                 \
    gat_bwd_src_kernel<W, C><<<grid, kThreads, 0, stream>>>(d_agg, num_nodes, colptr, row, cpos, ecoef, self_coef, d_h, \
                                                           d_a_src, d_out_mean, static_cast<__nv_bfloat16*>(d_h_hi), \
                                                           static_cast<__nv_bfloat16*>(d_h_lo));             \
  }
  ETPGT_DISPATCH_GAT(width, heads, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("gat_bwd");
  count_launch(1);
  return ETPGT_OK;
}

extern "C" int etpgt_gat_bwd(const float* h, const float* a_src, const float* a_dst, const float* d_agg,
                             const float* agg, int64_t num_nodes, int width, int heads, const int32_t* rowptr,
                             const int32_t* col, const int32_t* eperm, const int32_t* colptr, const int32_t* row,
                             const int32_t* cpos, int64_t num_edges, float negative_slope, const float* mask_edges,
                             const float* mask_self, const float* m, const float* inv_l, float* d_h,
                             float* d_a_src, float* d_a_dst, void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  ETPGT_REQUIRE(d_agg != nullptr, "gat_bwd: bad arguments");
  return etpgt_gat_bwd_mean(h, a_src, a_dst, d_agg, nullptr, agg, num_nodes, width, heads, rowptr, col, eperm, colptr,
                            row, cpos, num_edges, negative_slope, mask_edges, mask_self, m, inv_l, d_h, nullptr, nullptr,
                            d_a_src, d_a_dst, ws, ws_bytes, stream);
}

extern "C" int etpgt_sage_mean_fwd_split(const float* x, int64_t num_nodes, int dim, const int32_t* rowptr,
                                         const int32_t* col, float* mean, void* mean_hi, void* mean_lo, int64_t ld,
                                         etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(supported_dim(dim), "sage_mean_fwd: dim %d is not supported (dim must be one of 32, 64, 128, 256)",
                dim);
  ETPGT_REQUIRE(num_nodes >= 0 && x && rowptr && (mean || mean_hi) && (mean_hi == nullptr) == (mean_lo == nullptr),
                "sage_mean_fwd: bad arguments");
  ETPGT_REQUIRE(mean_hi == nullptr || (ld >= dim && ld % 4 == 0 && (((uintptr_t)mean_hi | (uintptr_t)mean_lo) & 7) == 0),
                "sage_mean_fwd: the split outputs need a pitch >= dim (multiple of 4) and 8-byte alignment");
  if (num_nodes == 0) return ETPGT_OK;
#define CALL(D)                                                                                              \
  {                                                                                                          \
    const int64_t npc = (kThreads / 32) * RowGeom<D>::GROUPS;                                                \
    sage_mean_fwd_kernel<D><<<(unsigned)((num_nodes + npc - 1) / npc), kThreads, 0, stream>>>(               \
        x, num_nodes, rowptr, col, mean, static_cast<__nv_bfloat16*>(mean_hi), static_cast<__nv_bfloat16*>(mean_lo), ld); \
  }
  ETPGT_DISPATCH_DIM(dim, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("sage_mean_fwd");
  return ETPGT_OK;
}

extern "C" int etpgt_sage_mean_fwd(const float* x, int64_t num_nodes, int dim, const int32_t* rowptr,
                                   const int32_t* col, float* mean, etpgt_stream_t stream) {
  ETPGT_REQUIRE(mean != nullptr, "sage_mean_fwd: bad arguments");
  return etpgt_sage_mean_fwd_split(x, num_nodes, dim, rowptr, col, mean, nullptr, nullptr, 0, stream);
}

extern "C" int etpgt_sage_mean_bwd_ld(const float* d_mean, int64_t ld, const float* d_root, int64_t num_nodes, int dim,
                                      const int32_t* rowptr, const int32_t* colptr, const int32_t* row, float* d_x,
                                      etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(supported_dim(dim), "sage_mean_bwd: dim %d is not supported (dim must be one of 32, 64, 128, 256)",
                dim);
  ETPGT_REQUIRE(num_nodes >= 0 && d_mean && rowptr && colptr && d_x && ld >= dim && ld % 4 == 0,
                "sage_mean_bwd: bad arguments");
  if (num_nodes == 0) return ETPGT_OK;
#define CALL(D)                                                                                              \
  {                                                                                                          \
    const int64_t npc = (kThreads / 32) * RowGeom<D>::GROUPS;                                                \
    sage_mean_bwd_kernel<D><<<(unsigned)((num_nodes + npc - 1) / npc), kThreads, 0, stream>>>(d_mean, ld, d_root, \
                                                                                             num_nodes, rowptr, colptr, \
                                                                                             row, d_x);      \
  }
  ETPGT_DISPATCH_DIM(dim, CALL)
#undef CALL
  ETPGT_CHECK_LAUNCH("sage_mean_bwd");
  return ETPGT_OK;
}

extern "C" int etpgt_sage_mean_bwd(const float* d_mean, int64_t num_nodes, int dim, const int32_t* rowptr,
                                   const int32_t* colptr, const int32_t* row, float* d_x, etpgt_stream_t stream) {
  return etpgt_sage_mean_bwd_ld(d_mean, dim, nullptr, num_nodes, dim, rowptr, colptr, row, d_x, stream);
}
