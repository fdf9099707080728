// Shared device/host helpers for the etpgt_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/etpgt_b200.h"

namespace etpgt {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this
constexpr int kWarp = 32;

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define ETPGT_REQUIRE(cond, ...)            \
  do {                                      \
    if (!(cond)) {                          \
      ::etpgt::set_error(__VA_ARGS__);      \
      return ETPGT_EINVAL;                  \
    }                                       \
  } while (0)

#define ETPGT_CHECK_LAUNCH(name)                                                  \
  do {                                                                            \
    cudaError_t e__ = cudaGetLastError();                                         \
    if (e__ != cudaSuccess) {                                                     \
      ::etpgt::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
      return ETPGT_ECUDA;                                                         \
    }                                                                             \
    ::etpgt::count_launch();                                                      \
  } while (0)

inline bool supported_dim(int dim) {
  return dim == 32 || dim == 64 || dim == 128 || dim == 256;
}
inline bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

// Bump allocator over the caller's workspace.
struct Workspace {
  char* base;
  size_t size;
  size_t used = 0;
  Workspace(void* p, size_t n) : base(static_cast<char*>(p)), size(n) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T));
    char* p = base + used;
    used += bytes;
    return reinterpret_cast<T*>(p);
  }
  bool ok() const { return used <= size; }
};

// grid for a persistent / grid-stride kernel: enough CTAs for `work` units but never more
// than `waves` CTAs per SM.
inline int grid_for(int64_t work_units, int units_per_cta, int ctas_per_sm) {
  int64_t want = (work_units + units_per_cta - 1) / units_per_cta;
  int64_t cap = static_cast<int64_t>(kNumSMs) * ctas_per_sm;
  if (want < 1) want = 1;
  return static_cast<int>(want < cap ? want : cap);
}

// ---------------------------------------------------------------------------- device side

// Row geometry: a feature row of DIM floats is spread over LPN lanes (a "group"), each lane
// holding V float4 registers; float4 slot v of lane l covers floats [4*(v*LPN+l), +4).
template <int DIM>
struct RowGeom {
  static constexpr int F4 = DIM / 4;                 // float4 per row
  static constexpr int LPN = F4 < 32 ? F4 : F4 % 32 == 0 ? 32 : 16;  // lanes per node (16 for DIM = 192)
  static constexpr int V = F4 / LPN;                 // float4 per lane
  static constexpr int GROUPS = 32 / LPN;            // nodes per warp
};

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
// streaming store: written once, read by a later kernel from L2/HBM, keep it out of L1
__device__ __forceinline__ void st4_stream(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }

__device__ __forceinline__ float dot4(float4 a, float4 b) { return a.x * b.x + a.y * b.y + a.z * b.z + a.w * b.w; }
__device__ __forceinline__ float4 fma4(float s, float4 a, float4 acc) {
  acc.x = fmaf(s, a.x, acc.x);
  acc.y = fmaf(s, a.y, acc.y);
  acc.z = fmaf(s, a.z, acc.z);
  acc.w = fmaf(s, a.w, acc.w);
  return acc;
}
__device__ __forceinline__ float4 scale4(float s, float4 a) { return make_float4(s * a.x, s * a.y, s * a.z, s * a.w); }
__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 sub4(float4 a, float4 b) { return make_float4(a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w); }
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

// butterfly sum over aligned groups of WIDTH lanes (WIDTH a power of two <= 32); every lane
// of the group ends with the group total.
template <int WIDTH>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int off = WIDTH / 2; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}
template <int WIDTH>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int off = WIDTH / 2; off > 0; off >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, off));
  return v;
}

// Per-head dot-product reduction for the row geometry above.
// part[v] holds this lane's partial dot over float4 slot v.  A head covers HEAD_F4 = C/4
// consecutive float4 of the row.  On return part[v] is the full dot product of the head that
// slot v of this lane belongs to.
template <int DIM, int HEAD_DIM>
__device__ __forceinline__ void head_reduce(float (&part)[RowGeom<DIM>::V]) {
  using G = RowGeom<DIM>;
  constexpr int HEAD_F4 = HEAD_DIM / 4;
  constexpr int SPAN = HEAD_F4 < G::LPN ? HEAD_F4 : G::LPN;  // lanes that share a head within a slot
#pragma unroll
  for (int v = 0; v < G::V; ++v) part[v] = group_sum<SPAN>(part[v]);
  if constexpr (HEAD_F4 > G::LPN) {
    constexpr int SLOTS = HEAD_F4 / G::LPN;  // consecutive slots per head
#pragma unroll
    for (int v0 = 0; v0 < G::V; v0 += SLOTS) {
      float s = 0.f;
#pragma unroll
      for (int u = 0; u < SLOTS; ++u) s += part[v0 + u];
#pragma unroll
      for (int u = 0; u < SLOTS; ++u) part[v0 + u] = s;
    }
  }
}

// head index of float4 slot v of lane `lane_in_group`
template <int DIM, int HEAD_DIM>
__device__ __forceinline__ int head_of(int v, int lane_in_group) {
  return (v * RowGeom<DIM>::LPN + lane_in_group) / (HEAD_DIM / 4);
}

// ---------------------------------------------------------------------------- Philox4x32-10
// Counter-based generator (Random123): the negative sampler (subgraph.cu) and the fused dropout of
// the BatchNorm epilogue (bn.cu) draw from it, keyed by (seed, element index), so a mask never has
// to be stored: forward and backward regenerate the same bits.
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
  c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
}
__device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
}
// Inverted-dropout factors of the four floats of float4 number `i4` of a tensor: 0 with probability
// p, else 1/(1-p).  threshold = p * 2^32 (host side); word w keeps its element iff w >= threshold.
__device__ __forceinline__ float4 dropout_factors4(uint64_t seed, uint64_t i4, uint32_t threshold, float keep_scale) {
  uint32_t c[4] = {(uint32_t)i4, (uint32_t)(i4 >> 32), 0x44524F50u /* "DROP" */, 0u};
  philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
  return make_float4(c[0] >= threshold ? keep_scale : 0.f, c[1] >= threshold ? keep_scale : 0.f,
                     c[2] >= threshold ? keep_scale : 0.f, c[3] >= threshold ? keep_scale : 0.f);
}
__device__ __forceinline__ float4 mul4(float4 a, float4 b) { return make_float4(a.x * b.x, a.y * b.y, a.z * b.z, a.w * b.w); }

}  // namespace etpgt

// Dispatch over the supported (dim, heads) pairs.  HEAD_DIM = dim / heads must be a power of
// two >= 4.  `KERNEL_CALL(DIM, HEAD_DIM)` is a statement.
#define ETPGT_DISPATCH_DIM(dim, CALL)   \
  switch (dim) {                        \
    case 32: { CALL(32); } break;       \
    case 64: { CALL(64); } break;       \
    case 128: { CALL(128); } break;     \
    case 256: { CALL(256); } break;     \
    default: break;                     \
  }

#define ETPGT_DH_CASE(D_, H_, CALL) \
  case (D_) * 16 + (H_): { CALL(D_, ((D_) / (H_))); } break;
#define ETPGT_DISPATCH_DIM_HEADS(dim, heads, CALL)                                   \
  switch ((dim) * 16 + (heads)) {                                                    \
    ETPGT_DH_CASE(32, 1, CALL) ETPGT_DH_CASE(32, 2, CALL) ETPGT_DH_CASE(32, 4, CALL) \
    ETPGT_DH_CASE(32, 8, CALL)                                                       \
    ETPGT_DH_CASE(64, 1, CALL) ETPGT_DH_CASE(64, 2, CALL) ETPGT_DH_CASE(64, 4, CALL) \
    ETPGT_DH_CASE(64, 8, CALL)                                                       \
    ETPGT_DH_CASE(128, 1, CALL) ETPGT_DH_CASE(128, 2, CALL) ETPGT_DH_CASE(128, 4, CALL) \
    ETPGT_DH_CASE(128, 8, CALL)                                                      \
    ETPGT_DH_CASE(256, 1, CALL) ETPGT_DH_CASE(256, 2, CALL) ETPGT_DH_CASE(256, 4, CALL) \
    ETPGT_DH_CASE(256, 8, CALL)                                                      \
    default:                                                                         \
      ::etpgt::set_error("unsupported (dim=%d, heads=%d): dim in {32,64,128,256}, heads in {1,2,4,8}", \
                         (int)(dim), (int)(heads));                                  \
      return ETPGT_EINVAL;                                                           \
  }
