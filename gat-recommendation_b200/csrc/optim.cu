// a11 / SURVEY.md §8(f1): the optimizer step of Trainer.train_epoch (etpgt/train/trainer.py:125-127) —
// torch.optim.AdamW(lr, weight_decay) built at scripts/train/train_baseline.py:252-256 and
// torch.optim.Adam(lr=1e-3) at scripts/pipeline/run_full_pipeline.py:210 — as ONE launch over every
// parameter of the model (the [num_items, 256] item table is 97 % of the bytes: 7 x 84 MB of traffic
// per step at 82k items, the largest byte mover of the step after the edge kernels).
//
// Dense decoupled-decay semantics of torch's single-tensor implementation, in its operation order:
//   AdamW:  p *= 1 - lr*wd                      Adam (L2):  g += wd * p
//   m  = m + (1-b1) * (g - m)                   (Tensor.lerp_)
//   v  = b2*v + (1-b2)*g*g                      (mul_ + addcmul_)
//   p -= (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
// bc1 = 1 - b1^step, bc2 = 1 - b2^step are computed by the caller in double (they are host scalars in
// torch too).  zero_grad != 0 also clears the gradient (the next backward ACCUMULATES rows into the same
// persistent buffer, so no separate 84 MB memset / add passes are needed).
//
// HBM-bound: 4 reads + 3 (4 with zero_grad) writes of 4 bytes per element; float4 accesses, chunked
// multi-tensor launch (one CTA = one 4,096-element chunk of one tensor).
#include <stdlib.h>

#include "peer.cuh"

namespace etpgt {
namespace {

constexpr int kThreads = 256;
constexpr int kChunk = 4096;       // elements per CTA: 4 float4 per thread in flight
constexpr int kMaxTensors = 48;    // per launch (kernel-parameter space)

struct AdamArgs {
  float* param[kMaxTensors];
  float* grad[kMaxTensors];
  float* exp_avg[kMaxTensors];
  float* exp_avg_sq[kMaxTensors];
  int64_t numel[kMaxTensors];
  int block_start[kMaxTensors + 1];  // first CTA of tensor t
  int count;
};

struct AdamScalars {
  float decay;        // AdamW: 1 - lr*wd;  Adam: wd
  float one_minus_b1, b1, b2, one_minus_b2, step_size, bc2_sqrt, eps;
  int decoupled, zero_grad, lerp_low;  // lerp_low: weight (1-b1) < 0.5, torch's first lerp formula
};

__device__ __forceinline__ void adam_one(float& p, float& g, float& m, float& v, const AdamScalars& s) {
  if (s.decoupled) p = p * s.decay;
  else g = fmaf(s.decay, p, g);
  m = s.lerp_low ? m + s.one_minus_b1 * (g - m) : g - (g - m) * s.b1;
  v = v * s.b2 + (s.one_minus_b2 * g) * g;
  const float denom = sqrtf(v) / s.bc2_sqrt + s.eps;
  p = p - (s.step_size * m) / denom;
}

__global__ void __launch_bounds__(kThreads)
adam_step_kernel(const __grid_constant__ AdamArgs a, const AdamScalars s) {
  // which tensor does this CTA belong to?  (<= 48 entries: a short scan, uniform over the CTA)
  int t = 0;
  while (t + 1 < a.count && (int)blockIdx.x >= a.block_start[t + 1]) ++t;
  const int64_t n = a.numel[t];
  const int64_t base = (int64_t)(blockIdx.x - a.block_start[t]) * kChunk;
  float* __restrict__ p = a.param[t];
  float* __restrict__ g = a.grad[t];
  float* __restrict__ m = a.exp_avg[t];
  float* __restrict__ v = a.exp_avg_sq[t];
  const bool vec = ((((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0) && base + kChunk <= n;
  if (vec) {
    float4 P[4], G[4], M[4], V[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t i = base + 4 * (u * kThreads + threadIdx.x);
      P[u] = ld4(p + i);
      G[u] = ld4(g + i);
      M[u] = ld4(m + i);
      V[u] = ld4(v + i);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      adam_one(P[u].x, G[u].x, M[u].x, V[u].x, s);
      adam_one(P[u].y, G[u].y, M[u].y, V[u].y, s);
      adam_one(P[u].z, G[u].z, M[u].z, V[u].z, s);
      adam_one(P[u].w, G[u].w, M[u].w, V[u].w, s);
      const int64_t i = base + 4 * (u * kThreads + threadIdx.x);
      st4(p + i, P[u]);
      st4(m + i, M[u]);
      st4(v + i, V[u]);
      if (s.zero_grad) st4(g + i, zero4());
    }
  } else {
    const int64_t end = base + kChunk < n ? base + kChunk : n;
    for (int64_t i = base + threadIdx.x; i < end; i += kThreads) {
      float P = p[i], G = g[i], M = m[i], V = v[i];
      adam_one(P, G, M, V, s);
      p[i] = P;
      m[i] = M;
      v[i] = V;
      if (s.zero_grad) g[i] = 0.f;
    }
  }
}

// Data parallelism over peer memory: reduce-scatter + AdamW + all-gather of the item table as ONE kernel.
// Rank `c.rank` owns the float4 range [begin4, end4) of the [rows, dim] table.  Per element it
//   * pulls that element of every rank's gradient buffer over NVLink and adds them in rank order (the
//     reduce-scatter; deterministic, so any owner would compute the same sum),
//   * applies the dense AdamW / Adam update with its own moments (only the owner keeps them current),
//   * pushes the new parameter value into every rank's copy of the table (the all-gather).
// Inbound (gradients) and outbound (parameters) traffic use opposite NVLink directions and overlap.
// The caller brackets the kernel with two communicator barriers: gradients complete before, every copy of
// the table complete (and every gradient buffer free to be cleared) after.
struct DpTableArgs {
  size_t param_offset, grad_offset;   // byte offsets of the table / its gradient inside every region
  float *exp_avg, *exp_avg_sq;        // this rank's moments, [rows, dim] (only the owned rows are touched)
  int64_t begin4, end4;
};

// UN elements per thread, ranks r < WMAX = 16 / UN: all UN * world gradient loads of a thread (up to 16 x 16 B,
// most of them over NVLink, ~2 us away) are in flight before the first one is used, so ONE CTA per SM (a quarter of
// its registers, no shared memory) keeps the links busy and leaves the SM to the kernels of the other stream (the
// exchange runs underneath the last phase of the backward pass).
template <int UN, int WMAX>
__global__ void __launch_bounds__(kThreads)
dp_adam_table_kernel(const __grid_constant__ CommView c, const DpTableArgs a, const AdamScalars s) {
  float4* __restrict__ m4 = reinterpret_cast<float4*>(a.exp_avg);
  float4* __restrict__ v4 = reinterpret_cast<float4*>(a.exp_avg_sq);
  const float4* p_own = reinterpret_cast<const float4*>(c.base[c.rank] + a.param_offset);
  const int64_t tile_elems = (int64_t)kThreads * UN;
  const int64_t tiles = (a.end4 - a.begin4 + tile_elems - 1) / tile_elems;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t first = a.begin4 + tile * tile_elems + threadIdx.x;
    float4 g[UN][WMAX];
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int64_t i = first + (int64_t)u * kThreads;
#pragma unroll
      for (int r = 0; r < WMAX; ++r)
        if (r < c.world && i < a.end4) g[u][r] = __ldcg(reinterpret_cast<const float4*>(c.base[r] + a.grad_offset) + i);
    }
#pragma unroll
    for (int u = 0; u < UN; ++u) {
      const int64_t i = first + (int64_t)u * kThreads;
      if (i >= a.end4) break;
      float4 P = p_own[i], M = m4[i], V = v4[i];
      float4 G = g[u][0];
#pragma unroll
      for (int r = 1; r < WMAX; ++r)
        if (r < c.world) G = add4(G, g[u][r]);      // rank order: every owner would form the same sum
      adam_one(P.x, G.x, M.x, V.x, s);
      adam_one(P.y, G.y, M.y, V.y, s);
      adam_one(P.z, G.z, M.z, V.z, s);
      adam_one(P.w, G.w, M.w, V.w, s);
#pragma unroll
      for (int r = 0; r < WMAX; ++r)
        if (r < c.world) reinterpret_cast<float4*>(c.base[r] + a.param_offset)[i] = P;
      m4[i] = M;
      v4[i] = V;
    }
  }
  __threadfence_system();   // the pushed rows are visible to the peers before this rank enters the barrier
}

bool fill_scalars(AdamScalars& s, double lr, double beta1, double beta2, double eps, double weight_decay,
                  int decoupled, int64_t step, int zero_grad) {
  // hyper-parameters arrive as doubles (Python floats in torch) and are rounded to fp32 only where
  // torch rounds them: 1 - beta is formed in double first
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  s.decay = (float)(decoupled ? 1.0 - lr * weight_decay : weight_decay);
  s.one_minus_b1 = (float)(1.0 - beta1);
  s.b2 = (float)beta2;
  s.one_minus_b2 = (float)(1.0 - beta2);
  s.step_size = (float)(lr / bc1);
  s.bc2_sqrt = (float)sqrt(bc2);
  s.b1 = (float)beta1;
  s.lerp_low = (1.0 - beta1) < 0.5;
  s.eps = (float)eps;
  s.decoupled = decoupled != 0;
  s.zero_grad = zero_grad != 0;
  return true;
}

// ---------------------------------------------------------------------------- row-sparse ("lazy") updates
// The item table's gradient touches only the rows of the batch (its items + negatives): at B = 1,024 and 82k
// items ~10 % of them.  These kernels read the whole gradient (4 B per element) but load, update and store
// p / m / v (and clear g) only for touched rows: rows * dim * 4 + touched * dim * 28 bytes instead of 32 per
// element.  A row is touched iff an element of its gradient row compares != 0 (+0 and -0 do not, NaN does).
// Listed mode (torch sparse gradients) instead updates every listed row, all-zero ones included.

// torch/optim/_functional.py::sparse_adam, one rounding per torch op (no FMA contraction):
//   mu = (g - m) * (1-b1);  m += mu;  vu = (g*g - v) * (1-b2);  v += vu
//   p += (-step_size) * ((mu + m_old) / (sqrt(vu + v_old) + eps))
struct SparseScalars {
  float one_minus_b1, one_minus_b2, neg_step_size, eps;
  int maximize;
};

__device__ __forceinline__ void sparse_adam_one(float& p, float g, float& m, float& v, const SparseScalars& s) {
  if (s.maximize) g = -g;
  const float mu = __fmul_rn(__fsub_rn(g, m), s.one_minus_b1);
  const float vu = __fmul_rn(__fsub_rn(__fmul_rn(g, g), v), s.one_minus_b2);
  const float numer = __fadd_rn(mu, m);
  const float denom = __fadd_rn(__fsqrt_rn(__fadd_rn(vu, v)), s.eps);
  m = __fadd_rn(m, mu);
  v = __fadd_rn(v, vu);
  p = __fadd_rn(p, __fmul_rn(__fdiv_rn(numer, denom), s.neg_step_size));
}

// adam_one outside the caller's data flow: inlined into a kernel, nvcc picks which of the two products of
// `v * b2 + (1-b2) * g * g` it contracts into an FMA from the surrounding code, and the row kernels for
// DIM <= 128 got the other one than adam_step_kernel (results 1 ulp apart).  Compiled once as its own function it
// takes adam_step_kernel's choice, so a touched row is bit-identical to the dense step.
struct AdamPMV {
  float p, m, v;
};
__device__ __noinline__ AdamPMV adam_one_isolated(float p, float g, float m, float v, const AdamScalars s) {
  adam_one(p, g, m, v, s);
  return {p, m, v};
}
struct AdamRowOp {
  AdamScalars s;
  __device__ __forceinline__ void operator()(float& p, float& g, float& m, float& v) const {
    const AdamPMV r = adam_one_isolated(p, g, m, v, s);
    p = r.p;
    m = r.m;
    v = r.v;
  }
};
struct SparseAdamRowOp {
  SparseScalars s;
  __device__ __forceinline__ void operator()(float& p, float& g, float& m, float& v) const {
    sparse_adam_one(p, g, m, v, s);
  }
};

constexpr int kRowThreads = 256;
constexpr int kRowCtasPerSM = 8;

struct RowArgs {
  float *param, *grad, *exp_avg, *exp_avg_sq;   // [rows, dim]; grad: [rows, dim] (scan) or [count, dim] (listed)
  const int64_t* index;                         // listed mode: table row of gradient row i
  int64_t rows, count;                          // count: gradient rows (scan: == rows)
  int dim, zero_grad;                           // zero_grad: clear touched gradient rows (scan mode)
  unsigned long long* touched;                  // optional: += rows updated
};

__device__ __forceinline__ bool nonzero4(float4 a) { return a.x != 0.f || a.y != 0.f || a.z != 0.f || a.w != 0.f; }

__device__ __forceinline__ void count_touched(unsigned n, unsigned long long* touched) {
  if (touched == nullptr) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(touched, (unsigned long long)n);
}

// DIM in {32, 64, 128, 256}: one lane group (RowGeom) per gradient row, grid-stride; float4 accesses (the caller
// checks 16-byte alignment).  The loop bound is warp-uniform, so every lane reaches the ballot.
template <int DIM, bool LISTED, class Op>
__global__ void __launch_bounds__(kRowThreads) adam_rows_kernel(const RowArgs a, const Op op) {
  using G = RowGeom<DIM>;
  const int lane = threadIdx.x & 31;
  const int grp = lane / G::LPN, lig = lane % G::LPN;
  const unsigned grp_mask = (G::LPN == 32 ? 0xffffffffu : ((1u << G::LPN) - 1u)) << (grp * G::LPN);
  const int64_t warp = ((int64_t)blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kRowThreads) >> 5;
  unsigned updated = 0;
  for (int64_t first = warp * G::GROUPS; first < a.count; first += nwarps * G::GROUPS) {
    const int64_t i = first + grp;
    int64_t row = i;
    bool live = i < a.count;
    if (LISTED && live) {
      row = a.index[i];
      live = row >= 0 && row < a.rows;
    }
    float4 g[G::V];
    bool nz = false;
    if (live) {
      const float* gr = a.grad + i * DIM;
#pragma unroll
      for (int v = 0; v < G::V; ++v) {
        g[v] = ld4(gr + 4 * (v * G::LPN + lig));
        nz |= nonzero4(g[v]);
      }
    }
    if ((__ballot_sync(0xffffffffu, LISTED ? live : nz) & grp_mask) == 0) continue;
    const int64_t off = row * DIM;
#pragma unroll
    for (int v = 0; v < G::V; ++v) {
      const int64_t e = off + 4 * (v * G::LPN + lig);
      float4 P = ld4(a.param + e), M = ld4(a.exp_avg + e), V = ld4(a.exp_avg_sq + e);
      op(P.x, g[v].x, M.x, V.x);
      op(P.y, g[v].y, M.y, V.y);
      op(P.z, g[v].z, M.z, V.z);
      op(P.w, g[v].w, M.w, V.w);
      st4(a.param + e, P);
      st4(a.exp_avg + e, M);
      st4(a.exp_avg_sq + e, V);
      if (!LISTED && a.zero_grad) st4(a.grad + i * DIM + 4 * (v * G::LPN + lig), zero4());
    }
    if (lig == 0) ++updated;
  }
  count_touched(updated, a.touched);
}

// any other dim: one warp per gradient row, scalar accesses
template <bool LISTED, class Op>
__global__ void __launch_bounds__(kRowThreads) adam_rows_scalar_kernel(const RowArgs a, const Op op) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * kRowThreads + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * kRowThreads) >> 5;
  const int64_t dim = a.dim;
  unsigned updated = 0;
  for (int64_t i = warp; i < a.count; i += nwarps) {
    int64_t row = i;
    if (LISTED) {
      row = a.index[i];
      if (row < 0 || row >= a.rows) continue;   // warp-uniform
    }
    float* gr = a.grad + i * dim;
    if (!LISTED) {
      bool nz = false;
      for (int64_t c = lane; c < dim; c += 32) nz |= gr[c] != 0.f;
      if (!__any_sync(0xffffffffu, nz)) continue;
    }
    const int64_t off = row * dim;
    for (int64_t c = lane; c < dim; c += 32) {
      float P = a.param[off + c], Gv = gr[c], M = a.exp_avg[off + c], V = a.exp_avg_sq[off + c];
      op(P, Gv, M, V);
      a.param[off + c] = P;
      a.exp_avg[off + c] = M;
      a.exp_avg_sq[off + c] = V;
      if (!LISTED && a.zero_grad) gr[c] = 0.f;
    }
    if (lane == 0) ++updated;
  }
  count_touched(updated, a.touched);
}

template <bool LISTED, class Op>
void launch_rows(const RowArgs& a, const Op& op, cudaStream_t stream) {
  const int rows_per_cta = (kRowThreads / 32) * (a.dim == 32 ? 4 : a.dim == 64 ? 2 : 1);
  const int grid = grid_for(a.count, rows_per_cta, kRowCtasPerSM);
  switch (a.dim) {
    case 32: adam_rows_kernel<32, LISTED><<<grid, kRowThreads, 0, stream>>>(a, op); break;
    case 64: adam_rows_kernel<64, LISTED><<<grid, kRowThreads, 0, stream>>>(a, op); break;
    case 128: adam_rows_kernel<128, LISTED><<<grid, kRowThreads, 0, stream>>>(a, op); break;
    case 256: adam_rows_kernel<256, LISTED><<<grid, kRowThreads, 0, stream>>>(a, op); break;
    default: adam_rows_scalar_kernel<LISTED><<<grid, kRowThreads, 0, stream>>>(a, op); break;
  }
}

bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" int etpgt_adam_step(const etpgt_adam_tensor* tensors, int count, double lr, double beta1, double beta2,
                               double eps, double weight_decay, int decoupled, int64_t step, int zero_grad,
                               etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(count >= 0 && (count == 0 || tensors != nullptr), "adam_step: bad tensor list");
  ETPGT_REQUIRE(step >= 1, "adam_step: step must be >= 1 (1-based, as torch counts it)");
  ETPGT_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0 && lr >= 0.0 &&
                    weight_decay >= 0.0,
                "adam_step: hyper-parameters out of range");
  for (int i = 0; i < count; ++i)
    ETPGT_REQUIRE(tensors[i].numel >= 0 && (tensors[i].numel == 0 || (tensors[i].param && tensors[i].grad &&
                                                                        tensors[i].exp_avg && tensors[i].exp_avg_sq)),
                  "adam_step: tensor %d has a NULL pointer", i);
  for (int i = 0; i < count; ++i)
    ETPGT_REQUIRE(tensors[i].numel < (int64_t(1) << 40), "adam_step: tensor %d too large", i);
  AdamScalars s;
  fill_scalars(s, lr, beta1, beta2, eps, weight_decay, decoupled, step, zero_grad);
  int done = 0;
  while (done < count) {
    AdamArgs a;
    a.count = 0;
    int blocks = 0;
    while (done < count && a.count < kMaxTensors) {
      const etpgt_adam_tensor& t = tensors[done++];
      if (t.numel == 0) continue;
      const int64_t nb = (t.numel + kChunk - 1) / kChunk;
      if (blocks + nb >= (int64_t(1) << 30)) { --done; break; }  // next launch
      a.param[a.count] = t.param;
      a.grad[a.count] = t.grad;
      a.exp_avg[a.count] = t.exp_avg;
      a.exp_avg_sq[a.count] = t.exp_avg_sq;
      a.numel[a.count] = t.numel;
      a.block_start[a.count] = blocks;
      blocks += (int)nb;
      ++a.count;
    }
    if (a.count == 0) break;
    a.block_start[a.count] = blocks;
    adam_step_kernel<<<blocks, kThreads, 0, stream>>>(a, s);
    ETPGT_CHECK_LAUNCH("adam_step");
  }
  return ETPGT_OK;
}

extern "C" int etpgt_dp_adam_table(const etpgt_comm_t* comm, size_t param_offset, size_t grad_offset, float* exp_avg,
                                   float* exp_avg_sq, int64_t rows, int dim, int64_t row_begin, int64_t row_end,
                                   double lr, double beta1, double beta2, double eps, double weight_decay,
                                   int decoupled, int64_t step, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(comm != nullptr, "dp_adam_table: null communicator");
  const CommView c = comm_view(comm);
  for (int r = 0; r < c.world; ++r) ETPGT_REQUIRE(c.base[r] != nullptr, "dp_adam_table: communicator not connected");
  ETPGT_REQUIRE(rows >= 0 && dim >= 4 && dim % 4 == 0 && row_begin >= 0 && row_begin <= row_end && row_end <= rows,
                "dp_adam_table: bad shape (rows %lld, dim %d, shard [%lld, %lld))", (long long)rows, dim,
                (long long)row_begin, (long long)row_end);
  ETPGT_REQUIRE(param_offset % 16 == 0 && grad_offset % 16 == 0 && exp_avg && exp_avg_sq &&
                    (((uintptr_t)exp_avg | (uintptr_t)exp_avg_sq) & 15) == 0,
                "dp_adam_table: buffers must be 16-byte aligned");
  ETPGT_REQUIRE(step >= 1 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0 && lr >= 0.0 &&
                    weight_decay >= 0.0,
                "dp_adam_table: hyper-parameters out of range");
  if (row_begin == row_end) return ETPGT_OK;
  AdamScalars s;
  fill_scalars(s, lr, beta1, beta2, eps, weight_decay, decoupled, step, 0);
  DpTableArgs a;
  a.param_offset = param_offset;
  a.grad_offset = grad_offset;
  a.exp_avg = exp_avg;
  a.exp_avg_sq = exp_avg_sq;
  a.begin4 = row_begin * (dim / 4);
  a.end4 = row_end * (dim / 4);
  // one CTA per SM: see the kernel's comment (ETPGT_DP_TABLE_CTAS: tuning knob for the grid)
  int cap = kNumSMs;
  if (const char* forced = getenv("ETPGT_DP_TABLE_CTAS")) {
    const int f = atoi(forced);
    if (f >= 1 && f <= 8 * kNumSMs) cap = f;
  }
  auto grid_of = [&](int un) {
    const int64_t tiles = (a.end4 - a.begin4 + (int64_t)kThreads * un - 1) / ((int64_t)kThreads * un);
    return (int)(tiles < cap ? tiles : cap);
  };
  if (c.world <= 2) {
    dp_adam_table_kernel<8, 2><<<grid_of(8), kThreads, 0, stream>>>(c, a, s);
  } else if (c.world <= 4) {
    dp_adam_table_kernel<4, 4><<<grid_of(4), kThreads, 0, stream>>>(c, a, s);
  } else {
    dp_adam_table_kernel<2, 8><<<grid_of(2), kThreads, 0, stream>>>(c, a, s);
  }
  ETPGT_CHECK_LAUNCH("dp_adam_table");
  return ETPGT_OK;
}

namespace {

int check_rows(const char* name, const float* param, const float* grad, const float* exp_avg,
               const float* exp_avg_sq, int64_t rows, int dim, int64_t step) {
  ETPGT_REQUIRE(rows >= 0 && dim >= 1 && rows < (int64_t(1) << 40) / dim, "%s: bad shape (rows %lld, dim %d)", name,
                (long long)rows, dim);
  ETPGT_REQUIRE(param && grad && exp_avg && exp_avg_sq, "%s: NULL pointer", name);
  ETPGT_REQUIRE(step >= 1, "%s: step must be >= 1 (1-based, as torch counts it)", name);
  ETPGT_REQUIRE(!supported_dim(dim) ||
                    (aligned16(param) && aligned16(grad) && aligned16(exp_avg) && aligned16(exp_avg_sq)),
                "%s: buffers must be 16-byte aligned for dim %d", name, dim);
  return ETPGT_OK;
}

}  // namespace

extern "C" int etpgt_adam_rows(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t rows, int dim,
                               double lr, double beta1, double beta2, double eps, double weight_decay, int decoupled,
                               int64_t step, int zero_grad, int64_t* touched, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int rc = check_rows("adam_rows", param, grad, exp_avg, exp_avg_sq, rows, dim, step);
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0 && lr >= 0.0 &&
                    weight_decay >= 0.0,
                "adam_rows: hyper-parameters out of range");
  if (touched && cudaMemsetAsync(touched, 0, sizeof(int64_t), stream) != cudaSuccess) {
    set_error("adam_rows: clearing the touched-row counter failed");
    return ETPGT_ECUDA;
  }
  if (rows == 0) return ETPGT_OK;
  AdamRowOp op;
  fill_scalars(op.s, lr, beta1, beta2, eps, weight_decay, decoupled, step, zero_grad);
  const RowArgs a{param, grad, exp_avg, exp_avg_sq, nullptr, rows, rows, dim, zero_grad != 0,
                  reinterpret_cast<unsigned long long*>(touched)};
  launch_rows<false>(a, op, stream);
  ETPGT_CHECK_LAUNCH("adam_rows");
  return ETPGT_OK;
}

extern "C" int etpgt_sparse_adam(float* param, float* exp_avg, float* exp_avg_sq, int64_t rows, int dim, float* grad,
                                 const int64_t* indices, int64_t nnz, double lr, double beta1, double beta2, double eps,
                                 int maximize, int64_t step, int zero_grad, int64_t* touched, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool listed = indices != nullptr;
  const int rc = check_rows("sparse_adam", param, grad, exp_avg, exp_avg_sq, rows, dim, step);
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(!listed || (nnz >= 0 && nnz < (int64_t(1) << 40) / dim),
                "sparse_adam: bad number of listed rows (%lld)", (long long)nnz);
  ETPGT_REQUIRE(!listed || zero_grad == 0, "sparse_adam: zero_grad applies to the dense (scan) mode only");
  ETPGT_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0 && lr >= 0.0,
                "sparse_adam: hyper-parameters out of range");
  if (touched && cudaMemsetAsync(touched, 0, sizeof(int64_t), stream) != cudaSuccess) {
    set_error("sparse_adam: clearing the touched-row counter failed");
    return ETPGT_ECUDA;
  }
  const int64_t count = listed ? nnz : rows;
  if (count == 0 || rows == 0) return ETPGT_OK;
  // constants as torch forms them: Python floats (double), rounded to fp32 where they meet the fp32 tensors
  const double bc1 = 1.0 - pow(beta1, (double)step);
  const double bc2 = 1.0 - pow(beta2, (double)step);
  SparseAdamRowOp op;
  op.s.one_minus_b1 = (float)(1.0 - beta1);
  op.s.one_minus_b2 = (float)(1.0 - beta2);
  op.s.neg_step_size = (float)(-(lr * sqrt(bc2) / bc1));
  op.s.eps = (float)eps;
  op.s.maximize = maximize != 0;
  const RowArgs a{param, grad, exp_avg, exp_avg_sq, indices, rows, count, dim, zero_grad != 0,
                  reinterpret_cast<unsigned long long*>(touched)};
  if (listed) launch_rows<true>(a, op, stream);
  else launch_rows<false>(a, op, stream);
  ETPGT_CHECK_LAUNCH("sparse_adam");
  return ETPGT_OK;
}
