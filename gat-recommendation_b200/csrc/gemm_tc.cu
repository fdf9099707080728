// Dense node projections on the tensor cores at fp32-grade accuracy ("split-bf16 x3").
//
// The per-layer projections of the path are fp32 nn.Linear GEMMs in the reference
// (TransformerConv lin_query/key/value/skip, PyG via graph_transformer.py:174): [N,256] x [256,1024].
// fp32 CUDA-core GEMMs were 62 % of the training step (profiles/r01_step_launches.txt).  Here every
// fp32 operand x is split as x = hi + lo (+ O(2^-18 |x|)), hi = bf16(x), lo = bf16(x - hi), and
//   C = A_hi B_hi^T + A_hi B_lo^T + A_lo B_hi^T        (fp32 accumulation in TMEM)
// is issued as three tcgen05.mma per k-step into the same accumulator: ~1e-5 relative error,
// inside the path's 1e-4 parity bound, at a third of the bf16 tensor rate instead of the fp32
// CUDA-core rate.  lo == NULL gives a plain bf16 GEMM.
//
//   etpgt_split_bf16      fp32 [R,C] -> hi/lo bf16 row-major and/or transposed (K-major operands
//                         for both the forward and the weight-gradient GEMM) + column sums
//   etpgt_gemm_bf16x3     C[M,N] = A[M,K] B[N,K]^T (+ bias[N]); persistent warp-specialised
//                         kernel on CTA pairs: TMA ring (A and B k-blocks, SWIZZLE_128B) -> tcgen05.mma
//                         256x128x16 or 256x256x16 (cta_group::2) -> multi-stage TMEM -> epilogue warps ->
//                         swizzled smem staging -> TMA tile stores (coalesced 128-byte rows, edges clipped);
//                         optional split-K with a fixed-order reduction (deterministic).
//
// Why CTA pairs: the GEMMs of a layer are bound by L2 -> shared-memory traffic (~1.6 GB in ~145 us each with one
// CTA per 128 x 128 tile = 11 TB/s at 50 % tensor-pipe activity), and a CTA working alone pulls its own copy of the
// B tile (in the forward projection all 148 CTAs reload the same 256 x 1024 weight matrix per k-block).  Here two CTAs
// on the two SMs of a TPC execute ONE tcgen05.mma of M = 256: each loads its own 128 rows of A and only HALF of the B
// tile, and the tensor cores of both SMs read both halves, so the B traffic per SM halves and a stage shrinks from 96
// to 64 KB (three stages instead of two at BN = 256).  Measured on the three GEMMs of one layer (M = 99,132, K or
// N = 256 / 1,024, split-bf16): forward / dX / dW 0.142 / 0.140 / 0.148 ms with one CTA per tile, 0.128 / 0.133 /
// 0.130 ms on pairs.
// Roles: warp 0 of BOTH CTAs is a TMA producer (its A rows, its B half; completion bytes are counted on the LEADER's
// full barrier, which expects two producer arrivals), warp 1 of the leader issues the MMAs and commits to the
// stage-empty / accumulator-full barriers of both CTAs (multicast commit), warps 2-5 of both CTAs drain their own 128
// accumulator rows from their own TMEM and release the accumulator stage on the leader's barrier (8 arrivals).
#include <math.h>

#include "tc_common.cuh"

namespace etpgt {
namespace {

using namespace tc;

constexpr int BLOCK_M = 128;
// Output tiles are 256 x BN per pair (128 x BN per CTA) with BN = 256 when N > 128, else 128 (template parameter,
// chosen per call by gemm_plan): the wider tile raises the flops per operand byte by a third.
constexpr int kTmemCols = 512;  // all of TMEM: 512 / BN accumulator stages
constexpr int kThreads = 192;  // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr uint32_t TILE_BYTES = BLOCK_M * BLOCK_K * 2;    // A: 16 KB per operand part per k-block
constexpr uint32_t MN_BOX_BYTES = 64 * BLOCK_K * 2;       // one 64(k) x 64(mn) box of an MN-major operand
constexpr int kEpiWarps = 4;
constexpr uint32_t CD_BOX_BYTES = 32 * 32 * 4;  // one 32-row x 32-column fp32 store box
constexpr uint32_t CD_BYTES = kEpiWarps * 2 * CD_BOX_BYTES;  // double-buffered per epilogue warp

struct __align__(8) GemmBarriers {
  uint64_t full[4];
  uint64_t empty[4];
  uint64_t acc_full[4];
  uint64_t acc_empty[4];
  uint32_t tmem_base;
};

// Optional second output of the epilogue (the FFN's first layer, etpgt/model/graph_transformer.py:109-124:
// Linear -> GELU -> Dropout): next to the fp32 pre-activation C (kept for the backward pass) the epilogue
// writes h = dropout(gelu(C)) directly as the split-bf16 operand pair of the next GEMM — the fp32 h and its
// split pass never exist.  GELU is the exact (erf) form of nn.GELU(); the dropout mask is Philox keyed by
// (seed, float4 index of the [M, N] tensor), the same bits etpgt_gelu_bwd_split regenerates.
struct ActEpilogue {
  __nv_bfloat16* hi;        // nullptr: no second output
  __nv_bfloat16* lo;
  int64_t ld;               // pitch of hi / lo in elements (multiple of 8)
  uint64_t seed;
  uint32_t drop_threshold;  // 0: no dropout
  float keep_scale;
};

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
// d/dx gelu(x) = Phi(x) + x phi(x)
__device__ __forceinline__ float gelu_grad(float x) {
  return 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x);
}

// eight consecutive output values of row `row` from column `col` on (col % 8 == 0)
__device__ __forceinline__ void act_store8(const ActEpilogue& act, float4 a, float4 b, int64_t row, int64_t col,
                                           int64_t N) {
  float x[8] = {gelu_exact(a.x), gelu_exact(a.y), gelu_exact(a.z), gelu_exact(a.w),
                gelu_exact(b.x), gelu_exact(b.y), gelu_exact(b.z), gelu_exact(b.w)};
  if (act.drop_threshold != 0) {
    const uint64_t i4 = (uint64_t)(row * N + col) >> 2;
    const float4 f0 = dropout_factors4(act.seed, i4, act.drop_threshold, act.keep_scale);
    const float4 f1 = dropout_factors4(act.seed, i4 + 1, act.drop_threshold, act.keep_scale);
    x[0] *= f0.x; x[1] *= f0.y; x[2] *= f0.z; x[3] *= f0.w;
    x[4] *= f1.x; x[5] *= f1.y; x[6] *= f1.z; x[7] *= f1.w;
  }
  uint32_t h[4], l[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const __nv_bfloat16 h0 = __float2bfloat16_rn(x[2 * t]), h1 = __float2bfloat16_rn(x[2 * t + 1]);
    const __nv_bfloat16 l0 = __float2bfloat16_rn(x[2 * t] - __bfloat162float(h0));
    const __nv_bfloat16 l1 = __float2bfloat16_rn(x[2 * t + 1] - __bfloat162float(h1));
    h[t] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
    l[t] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
  }
  *reinterpret_cast<uint4*>(act.hi + row * act.ld + col) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(act.lo + row * act.ld + col) = make_uint4(l[0], l[1], l[2], l[3]);
}

// PARTS = 1: plain bf16 (A_hi, B_hi).  PARTS = 2: split operands, three products.
template <int PARTS, int BN> struct StageCount2 {          // ring depth that fits 227 KB next to the store boxes
  static constexpr int value = PARTS == 2 ? (BN == 256 ? 3 : 4) : 4;
};

template <int PARTS, int BLOCK_N>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16x3_2sm_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                       const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
                       const __grid_constant__ CUtensorMap map_c /* C, or the [split_k][M][N] partials */,
                       int64_t M, int64_t N, int64_t K, int m_pairs, int n_tiles, int split_k, int kb_per_split,
                       const float* __restrict__ bias, int a_mn, int b_mn, int accumulate, const ActEpilogue act) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  constexpr int kStages = StageCount2<PARTS, BLOCK_N>::value;
  constexpr int kAccStages = kTmemCols / BLOCK_N;
  constexpr int HALF_N = BLOCK_N / 2;
  constexpr uint32_t B_HALF_BYTES = HALF_N * BLOCK_K * 2;   // this CTA's half of B: 8 / 16 KB per part per k-block
  constexpr uint32_t kInstrDesc = instr_desc_bf16(2 * BLOCK_M, BLOCK_N);
  constexpr uint32_t STAGE_BYTES = PARTS * (TILE_BYTES + B_HALF_BYTES);
  uint8_t* smem_cd = smem + kStages * STAGE_BYTES;
  GemmBarriers* bars = reinterpret_cast<GemmBarriers*>(smem_cd + CD_BYTES);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();          // 0 = leader
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int total_kb = (int)((K + BLOCK_K - 1) / BLOCK_K);
  const int64_t total_units = (int64_t)m_pairs * n_tiles * split_k;

  if (threadIdx.x == 0) {
    for (int s = 0; s < 4; ++s) { mbar_init(&bars->full[s], 2); mbar_init(&bars->empty[s], 1); }
    for (int s = 0; s < 4; ++s) { mbar_init(&bars->acc_full[s], 1); mbar_init(&bars->acc_empty[s], 2 * kEpiWarps); }
    fence_barrier_init();
    tma_prefetch_desc(&map_a_hi);
    tma_prefetch_desc(&map_b_hi);
    tma_prefetch_desc(&map_c);
    if (PARTS == 2) { tma_prefetch_desc(&map_a_lo); tma_prefetch_desc(&map_b_lo); }
  }
  if (warp == 1) tmem_alloc_2sm(&bars->tmem_base, kTmemCols);
  tc_fence_before();
  cluster_sync_all();        // both CTAs' barriers are initialised before anything crosses the pair
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  auto decode = [&](int64_t u, int& ks, int& mp, int& nt) {
    nt = (int)(u % n_tiles);
    mp = (int)((u / n_tiles) % m_pairs);
    ks = (int)(u / ((int64_t)n_tiles * m_pairs));
  };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int64_t u = pair; u < total_units; u += num_pairs) {
        int ks, mp, nt;
        decode(u, ks, mp, nt);
        const int kb0 = ks * kb_per_split;
        const int kb1 = kb0 + kb_per_split < total_kb ? kb0 + kb_per_split : total_kb;
        const int m0 = (2 * mp + (int)rank) * BLOCK_M;           // this CTA's rows of A / C
        const int n0 = nt * BLOCK_N + (int)rank * HALF_N;        // this CTA's half of the B tile
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          const uint32_t full = mapa_shared(smem_u32(&bars->full[stage]), 0);   // the leader's barrier
          mbar_arrive_expect_tx_cluster(full, STAGE_BYTES);
          uint8_t* st = smem + stage * STAGE_BYTES;
          auto load = [&](const CUtensorMap* map, uint8_t* dst, int mn0, int mn_major, int rows) {
            if (mn_major) {
              for (int b = 0; b < rows / 64; ++b)
                tma_load_2d_2sm(map, full, dst + b * MN_BOX_BYTES, mn0 + 64 * b, kb * BLOCK_K);
            } else {
              tma_load_2d_2sm(map, full, dst, kb * BLOCK_K, mn0);
            }
          };
          load(&map_a_hi, st, m0, a_mn, BLOCK_M);
          if (PARTS == 2) load(&map_a_lo, st + TILE_BYTES, m0, a_mn, BLOCK_M);
          load(&map_b_hi, st + PARTS * TILE_BYTES, n0, b_mn, HALF_N);
          if (PARTS == 2) load(&map_b_lo, st + PARTS * TILE_BYTES + B_HALF_BYTES, n0, b_mn, HALF_N);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int t = 0;
      const uint32_t idesc = kInstrDesc | (a_mn ? 1u << 15 : 0u) | (b_mn ? 1u << 16 : 0u);
      for (int64_t u = pair; u < total_units; u += num_pairs, ++t) {
        int ks, mp, nt;
        decode(u, ks, mp, nt);
        const int kb0 = ks * kb_per_split;
        const int kb1 = kb0 + kb_per_split < total_kb ? kb0 + kb_per_split : total_kb;
        const int acc = t % kAccStages;
        mbar_wait(&bars->acc_empty[acc], ((uint32_t)(t / kAccStages) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after();
          const uint32_t a_hi = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t a_lo = a_hi + TILE_BYTES;
          const uint32_t b_hi = a_hi + PARTS * TILE_BYTES;
          const uint32_t b_lo = b_hi + B_HALF_BYTES;
#pragma unroll
          for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
            const uint32_t off_a = a_mn ? kk * UMMA_K * 128 : kk * UMMA_K * 2;
            const uint32_t off_b = b_mn ? kk * UMMA_K * 128 : kk * UMMA_K * 2;
            const uint32_t first = (kb == kb0 && kk == 0) ? 0u : 1u;
            const uint64_t da_hi = a_mn ? make_desc_mn_sw128(a_hi + off_a, MN_BOX_BYTES) : make_desc_sw128(a_hi + off_a);
            const uint64_t db_hi = b_mn ? make_desc_mn_sw128(b_hi + off_b, MN_BOX_BYTES) : make_desc_sw128(b_hi + off_b);
            umma_bf16_2sm(tmem_d, da_hi, db_hi, idesc, first);
            if (PARTS == 2) {
              const uint64_t da_lo = a_mn ? make_desc_mn_sw128(a_lo + off_a, MN_BOX_BYTES) : make_desc_sw128(a_lo + off_a);
              const uint64_t db_lo = b_mn ? make_desc_mn_sw128(b_lo + off_b, MN_BOX_BYTES) : make_desc_sw128(b_lo + off_b);
              umma_bf16_2sm(tmem_d, da_hi, db_lo, idesc, 1u);
              umma_bf16_2sm(tmem_d, da_lo, db_hi, idesc, 1u);
            }
          }
          umma_commit_2sm(&bars->empty[stage]);      // the stage is free in BOTH CTAs
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit_2sm(&bars->acc_full[acc]);       // both CTAs' epilogues may read their accumulator rows
      }
    }
  } else {
    const int quarter = warp & 3;
    uint8_t* my_cd = smem_cd + (warp - 2) * 2 * CD_BOX_BYTES;
    const bool add_bias = bias != nullptr && split_k == 1;
    int buf = 0;
    int t = 0;
    for (int64_t u = pair; u < total_units; u += num_pairs, ++t) {
      int ks, mp, nt;
      decode(u, ks, mp, nt);
      const int acc = t % kAccStages;
      mbar_wait(&bars->acc_full[acc], (uint32_t)(t / kAccStages) & 1);
      tc_fence_after();
      const int row0 = (2 * mp + (int)rank) * BLOCK_M + quarter * 32;
      const int col0 = nt * BLOCK_N;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BLOCK_N);
#pragma unroll 1
      for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
        float4 bv[8];
        const bool bias_on = add_bias && (int64_t)col0 + c0 + 32 <= N;
        if (bias_on) {
#pragma unroll
          for (int j = 0; j < 8; ++j) bv[j] = ldg4(bias + col0 + c0 + 4 * j);
        }
        uint32_t v[32];
        tmem_ld_32x32(taddr + (uint32_t)c0, v);
        if (c0 + 32 == BLOCK_N) {  // accumulator fully read: release the stage on the LEADER's barrier
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&bars->acc_empty[acc]), 0));
        }
        if ((int64_t)col0 + c0 >= N || row0 >= M) continue;  // whole chunk outside the matrix (warp-uniform)
        if (lane == 0) tma_store_wait_read<1>();
        __syncwarp();
        uint8_t* box = my_cd + buf * CD_BOX_BYTES + lane * 128;
        float4 prev = zero4();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float4 o = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                 __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
          const int64_t col = (int64_t)col0 + c0 + 4 * j;
          if (bias_on) o = add4(o, bv[j]);
          else if (add_bias && col + 3 < N) o = add4(o, ldg4(bias + col));
          *reinterpret_cast<float4*>(box + ((j ^ (lane & 7)) << 4)) = o;
          if (act.hi != nullptr) {   // warp-uniform
            if (j & 1) { if (row0 + lane < M && col + 3 < N) act_store8(act, prev, o, row0 + lane, col - 4, N); }
            else prev = o;
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          if (accumulate && split_k == 1) tma_reduce_add_3d(&map_c, my_cd + buf * CD_BOX_BYTES, col0 + c0, row0, 0);
          else tma_store_3d(&map_c, my_cd + buf * CD_BOX_BYTES, col0 + c0, row0, split_k > 1 ? ks : 0);
          tma_store_commit();
        }
        buf ^= 1;
      }
    }
    if (lane == 0) tma_store_wait_all();
  }
  tc_fence_before();
  cluster_sync_all();        // neither CTA's shared memory / TMEM goes away while the other still uses it
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, kTmemCols);
  }
}

// C[m][n] = bias[n] + sum_s partial[s][m][n], s ascending: deterministic split-K reduction.
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ partial, int split_k, int64_t M, int64_t N,
                     const float* __restrict__ bias, float* __restrict__ C, int64_t ldc, int accumulate) {
  const int64_t total4 = M * N / 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = (4 * i) / N, n = (4 * i) % N;
    float4 acc = bias != nullptr ? ldg4(bias + n) : zero4();
    if (accumulate) acc = add4(acc, ld4(C + m * ldc + n));
    for (int s = 0; s < split_k; ++s) acc = add4(acc, ldg4(partial + ((int64_t)s * M + m) * N + n));
    st4(C + m * ldc + n, acc);
  }
}

// ------------------------------------------------------------------------------ split kernel
// 64 x 64 fp32 tile per CTA (256 threads): row-major hi/lo written straight from the coalesced
// read, transposed hi/lo through a padded shared-memory tile, column sums as per-CTA partials.
constexpr int SPLIT_TILE = 64;

__device__ __forceinline__ void split_one(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(x);
  lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

__global__ void __launch_bounds__(256)
split_bf16_kernel(const float* __restrict__ src, int64_t rows, int64_t cols, int64_t ld_src,
                  __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, int64_t ld_out,
                  __nv_bfloat16* __restrict__ hi_t, __nv_bfloat16* __restrict__ lo_t, int64_t ld_t,
                  float* __restrict__ colsum_partial /* [row_tiles][cols] */) {
  __shared__ float tile[SPLIT_TILE][SPLIT_TILE + 1];
  const int64_t r0 = (int64_t)blockIdx.y * SPLIT_TILE, c0 = (int64_t)blockIdx.x * SPLIT_TILE;
  const int tx = threadIdx.x % SPLIT_TILE, ty = threadIdx.x / SPLIT_TILE;  // 64 x 4
  for (int rr = ty; rr < SPLIT_TILE; rr += 4) {
    const int64_t r = r0 + rr, c = c0 + tx;
    float x = 0.f;
    if (r < rows && c < cols) {
      x = src[r * ld_src + c];
      if (hi != nullptr) {
        __nv_bfloat16 h, l;
        split_one(x, h, l);
        hi[r * ld_out + c] = h;
        if (lo != nullptr) lo[r * ld_out + c] = l;
      }
    }
    tile[rr][tx] = x;
  }
  __syncthreads();
  if (hi_t != nullptr) {
    for (int cc = ty; cc < SPLIT_TILE; cc += 4) {
      const int64_t c = c0 + cc, r = r0 + tx;
      if (c < cols && r < rows) {
        __nv_bfloat16 h, l;
        split_one(tile[tx][cc], h, l);
        hi_t[c * ld_t + r] = h;
        if (lo_t != nullptr) lo_t[c * ld_t + r] = l;
      }
    }
  }
  if (colsum_partial != nullptr && threadIdx.x < SPLIT_TILE) {
    const int64_t c = c0 + threadIdx.x;
    if (c < cols) {
      float s = 0.f;
      for (int rr = 0; rr < SPLIT_TILE; ++rr) s += tile[rr][threadIdx.x];
      colsum_partial[(int64_t)blockIdx.y * cols + c] = s;
    }
  }
}

// Backward of the FFN's Linear -> GELU -> Dropout (the forward is the ActEpilogue of the GEMM):
// du = d_h * dropout_factor * gelu'(u), written directly as the split-bf16 operand pair of the two weight / input
// gradient GEMMs, with its column sums (the first layer's bias gradient) as per-CTA partials.
__global__ void __launch_bounds__(256)
gelu_bwd_split_kernel(const float* __restrict__ d_h, const float* __restrict__ u, int64_t rows, int64_t cols,
                      uint64_t seed, uint32_t drop_threshold, float keep_scale, __nv_bfloat16* __restrict__ hi,
                      __nv_bfloat16* __restrict__ lo, int64_t ld_out, float* __restrict__ colsum_partial) {
  __shared__ float tile[SPLIT_TILE][SPLIT_TILE + 1];
  const int64_t r0 = (int64_t)blockIdx.y * SPLIT_TILE, c0 = (int64_t)blockIdx.x * SPLIT_TILE;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;  // 16 float4 columns x 16 rows
  for (int rr = ty; rr < SPLIT_TILE; rr += 16) {
    const int64_t r = r0 + rr, c = c0 + 4 * tx;
    float4 x = zero4();
    if (r < rows && c < cols) {
      const float4 g = ldg4(d_h + r * cols + c), uv = ldg4(u + r * cols + c);
      x = make_float4(g.x * gelu_grad(uv.x), g.y * gelu_grad(uv.y), g.z * gelu_grad(uv.z), g.w * gelu_grad(uv.w));
      if (drop_threshold != 0) x = mul4(x, dropout_factors4(seed, (uint64_t)(r * cols + c) >> 2, drop_threshold, keep_scale));
      const float e[4] = {x.x, x.y, x.z, x.w};
      uint32_t h2[2], l2[2];
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        __nv_bfloat16 h0, l0, h1, l1;
        split_one(e[2 * t], h0, l0);
        split_one(e[2 * t + 1], h1, l1);
        h2[t] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
        l2[t] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
      }
      *reinterpret_cast<uint2*>(hi + r * ld_out + c) = make_uint2(h2[0], h2[1]);
      *reinterpret_cast<uint2*>(lo + r * ld_out + c) = make_uint2(l2[0], l2[1]);
    }
    tile[rr][4 * tx] = x.x; tile[rr][4 * tx + 1] = x.y; tile[rr][4 * tx + 2] = x.z; tile[rr][4 * tx + 3] = x.w;
  }
  __syncthreads();
  if (colsum_partial != nullptr && threadIdx.x < SPLIT_TILE) {
    const int64_t c = c0 + threadIdx.x;
    if (c < cols) {
      float s = 0.f;
      for (int rr = 0; rr < SPLIT_TILE; ++rr) s += tile[rr][threadIdx.x];
      colsum_partial[(int64_t)blockIdx.y * cols + c] = s;
    }
  }
}

// one warp per output column, lanes stride over the row tiles, fixed butterfly: deterministic
__global__ void __launch_bounds__(256)
colsum_reduce_kernel(const float* __restrict__ partial, int64_t parts, int64_t cols, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t c = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (c >= cols) return;
  float s = 0.f;
  for (int64_t p = lane; p < parts; p += 32) s += partial[p * cols + c];
  s = group_sum<32>(s);
  if (lane == 0) out[c] = s;
}

struct GemmPlan {
  int m_tiles, n_tiles, split_k, kb_per_split, grid, block_n;   // m_tiles counts 256-row pair tiles; grid = 2 x pairs
};

GemmPlan gemm_plan(int64_t M, int64_t N, int64_t K, int want_split) {
  GemmPlan p;
  p.block_n = N > 128 ? 256 : 128;   // see the note at the top
  p.m_tiles = (int)((M + 2 * BLOCK_M - 1) / (2 * BLOCK_M));
  p.n_tiles = (int)((N + p.block_n - 1) / p.block_n);
  const int total_kb = (int)((K + BLOCK_K - 1) / BLOCK_K);
  const int workers = kNumSMs / 2;   // SM pairs
  int split = 1;
  if (want_split != 1) {
    // few output tiles and a long K: split K until about two waves of units exist
    const int64_t tiles = (int64_t)p.m_tiles * p.n_tiles;
    if (tiles < workers && total_kb >= 16) {
      split = (int)((2 * workers + tiles - 1) / tiles);
      if (split > total_kb / 8) split = total_kb / 8;
      if (split < 1) split = 1;
    }
    if (want_split > 1) split = want_split;
  }
  p.kb_per_split = (total_kb + split - 1) / split;
  p.split_k = (total_kb + p.kb_per_split - 1) / p.kb_per_split;
  const int64_t units = (int64_t)p.m_tiles * p.n_tiles * p.split_k;
  p.grid = 2 * (int)(units < workers ? units : workers);
  if (p.grid < 2) p.grid = 2;
  return p;
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_split_bf16_workspace_bytes(int64_t rows, int64_t cols) {
  const int64_t row_tiles = (rows + SPLIT_TILE - 1) / SPLIT_TILE;
  return align_up((size_t)(row_tiles > 0 ? row_tiles : 1) * cols * sizeof(float)) + 256;
}

extern "C" int etpgt_split_bf16(const float* src, int64_t rows, int64_t cols, int64_t ld_src, void* hi, void* lo,
                                int64_t ld_out, void* hi_t, void* lo_t, int64_t ld_t, float* colsum, void* ws,
                                size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(rows >= 0 && cols > 0 && ld_src >= cols, "split_bf16: bad sizes");
  ETPGT_REQUIRE(hi == nullptr || ld_out >= cols, "split_bf16: ld_out < cols");
  ETPGT_REQUIRE(hi_t == nullptr || ld_t >= rows, "split_bf16: ld_t < rows");
  ETPGT_REQUIRE(lo == nullptr || hi != nullptr, "split_bf16: lo without hi");
  ETPGT_REQUIRE(lo_t == nullptr || hi_t != nullptr, "split_bf16: lo_t without hi_t");
  if (colsum != nullptr && ws_bytes < etpgt_split_bf16_workspace_bytes(rows, cols)) {
    set_error("split_bf16: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  const int64_t row_tiles = (rows + SPLIT_TILE - 1) / SPLIT_TILE, col_tiles = (cols + SPLIT_TILE - 1) / SPLIT_TILE;
  float* partial = colsum != nullptr ? static_cast<float*>(ws) : nullptr;
  if (rows > 0) {
    split_bf16_kernel<<<dim3((unsigned)col_tiles, (unsigned)row_tiles), 256, 0, stream>>>(
        src, rows, cols, ld_src, static_cast<__nv_bfloat16*>(hi), static_cast<__nv_bfloat16*>(lo), ld_out,
        static_cast<__nv_bfloat16*>(hi_t), static_cast<__nv_bfloat16*>(lo_t), ld_t, partial);
    ETPGT_CHECK_LAUNCH("split_bf16");
  }
  if (colsum != nullptr) {
    colsum_reduce_kernel<<<(unsigned)((cols * 32 + 255) / 256), 256, 0, stream>>>(partial, rows > 0 ? row_tiles : 0, cols,
                                                                                 colsum);
    ETPGT_CHECK_LAUNCH("colsum_reduce");
  }
  return ETPGT_OK;
}

extern "C" size_t etpgt_gemm_bf16x3_workspace_bytes(int64_t M, int64_t N, int64_t K, int split_k) {
  const GemmPlan p = gemm_plan(M, N, K, split_k);
  return (p.split_k > 1 ? align_up((size_t)p.split_k * M * N * sizeof(float)) : 0) + 256;
}

static int gemm_run(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, int64_t M, int64_t N,
                    int64_t K, int64_t lda, int64_t ldb, int a_mn_major, int b_mn_major, const float* bias,
                    int accumulate, float* C, int64_t ldc, int split_k, void* ws, size_t ws_bytes,
                    etpgt_stream_t stream_, const ActEpilogue& act) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(M >= 0 && N > 0 && K > 0 && M < (int64_t(1) << 31) && N < (int64_t(1) << 31) && K < (int64_t(1) << 31),
                "gemm_bf16x3: bad sizes");
  ETPGT_REQUIRE(a_hi && b_hi && C && (a_lo == nullptr) == (b_lo == nullptr),
                "gemm_bf16x3: operands: hi parts required, lo parts both or neither");
  ETPGT_REQUIRE(lda >= (a_mn_major ? M : K) && ldb >= (b_mn_major ? N : K) && lda % 8 == 0 && ldb % 8 == 0,
                "gemm_bf16x3: operand pitches must cover the contiguous extent and be multiples of 8 elements");
  ETPGT_REQUIRE(N % 4 == 0 && ldc % 4 == 0 && ldc >= N, "gemm_bf16x3: N and ldc must be multiples of 4");
  ETPGT_REQUIRE((((uintptr_t)a_hi | (uintptr_t)b_hi | (uintptr_t)a_lo | (uintptr_t)b_lo | (uintptr_t)C) & 15) == 0,
                "gemm_bf16x3: pointers must be 16-byte aligned");
  if (M == 0) return ETPGT_OK;
  const GemmPlan p = gemm_plan(M, N, K, split_k);
  if (ws_bytes < etpgt_gemm_bf16x3_workspace_bytes(M, N, K, split_k)) {
    set_error("gemm_bf16x3: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  // K-major operand [MN, K]: boxes of 128 (A) / BN / 2 (B: this CTA's half) rows x 64 k.  MN-major operand [K, MN]: boxes of 64 k-rows x 64 mn.
  auto map_a = [&](CUtensorMap* m, const void* ptr_) {
    return a_mn_major ? make_map_bf16(m, ptr_, K, M, lda, 64) : make_map_bf16(m, ptr_, M, K, lda, BLOCK_M);
  };
  auto map_b = [&](CUtensorMap* m, const void* ptr_) {
    return b_mn_major ? make_map_bf16(m, ptr_, K, N, ldb, 64)
                      : make_map_bf16(m, ptr_, N, K, ldb, p.block_n / 2);
  };
  bool ok = map_a(&ma_hi, a_hi) && map_b(&mb_hi, b_hi);
  if (a_lo != nullptr) ok = ok && map_a(&ma_lo, a_lo) && map_b(&mb_lo, b_lo);
  else { ma_lo = ma_hi; mb_lo = mb_hi; }
  if (!ok) {
    set_error("gemm_bf16x3: cuTensorMapEncodeTiled failed");
    return ETPGT_ECUDA;
  }
  float* partial = p.split_k > 1 ? static_cast<float*>(ws) : nullptr;
  CUtensorMap mc;
  if (!(p.split_k > 1 ? make_map_f32_store(&mc, partial, p.split_k, M, N, N, M * N)
                      : make_map_f32_store(&mc, C, 1, M, N, ldc, M * ldc))) {
    set_error("gemm_bf16x3: cuTensorMapEncodeTiled (output) failed");
    return ETPGT_ECUDA;
  }
  const int parts = a_lo != nullptr ? 2 : 1;
#define LAUNCH(PARTS_, BN_)                                                                                       \
  {                                                                                                               \
    const size_t smem = 1024 + (size_t)StageCount2<PARTS_, BN_>::value * PARTS_ * (TILE_BYTES + BN_ / 2 * BLOCK_K * 2) + \
                        CD_BYTES + sizeof(GemmBarriers) + 64;                                                     \
    cudaFuncSetAttribute(gemm_bf16x3_2sm_kernel<PARTS_, BN_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    cudaLaunchConfig_t cfg = {};                                                                                  \
    cfg.gridDim = dim3(p.grid);                                                                                   \
    cfg.blockDim = dim3(kThreads);                                                                                \
    cfg.dynamicSmemBytes = smem;                                                                                  \
    cfg.stream = stream;                                                                                          \
    cudaLaunchAttribute attr[1];                                                                                  \
    attr[0].id = cudaLaunchAttributeClusterDimension;                                                             \
    attr[0].val.clusterDim.x = 2;                                                                                 \
    attr[0].val.clusterDim.y = 1;                                                                                 \
    attr[0].val.clusterDim.z = 1;                                                                                 \
    cfg.attrs = attr;                                                                                             \
    cfg.numAttrs = 1;                                                                                             \
    cudaLaunchKernelEx(&cfg, gemm_bf16x3_2sm_kernel<PARTS_, BN_>, ma_hi, ma_lo, mb_hi, mb_lo, mc, M, N, K,        \
                       p.m_tiles, p.n_tiles, p.split_k, p.kb_per_split, bias, (int)(a_mn_major != 0),             \
                       (int)(b_mn_major != 0), (int)(accumulate != 0), act);                                      \
  }
  if (parts == 2 && p.block_n == 256) LAUNCH(2, 256)
  else if (parts == 2) LAUNCH(2, 128)
  else if (p.block_n == 256) LAUNCH(1, 256)
  else LAUNCH(1, 128)
#undef LAUNCH
  ETPGT_CHECK_LAUNCH("gemm_bf16x3");
  if (p.split_k > 1) {
    splitk_reduce_kernel<<<grid_for(M * N / 4, 256 * 2, 8), 256, 0, stream>>>(partial, p.split_k, M, N, bias, C, ldc,
                                                                              accumulate != 0);
    ETPGT_CHECK_LAUNCH("splitk_reduce");
  }
  return ETPGT_OK;
}

extern "C" int etpgt_gemm_bf16x3_ex(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, int64_t M,
                                    int64_t N, int64_t K, int64_t lda, int64_t ldb, int a_mn_major, int b_mn_major,
                                    const float* bias, int accumulate, float* C, int64_t ldc, int split_k, void* ws,
                                    size_t ws_bytes, etpgt_stream_t stream) {
  ActEpilogue none = {};
  return gemm_run(a_hi, a_lo, b_hi, b_lo, M, N, K, lda, ldb, a_mn_major, b_mn_major, bias, accumulate, C, ldc, split_k,
                  ws, ws_bytes, stream, none);
}

// p -> (threshold = p * 2^32, scale = 1 / (1 - p)); p == 0 disables the mask (the same mapping as bn.cu)
static bool gelu_dropout_params(double p, uint32_t* threshold, float* keep_scale) {
  if (!(p >= 0.0 && p < 1.0)) return false;
  const double t = p * 4294967296.0;
  *threshold = p > 0.0 ? (uint32_t)(t < 1.0 ? 1.0 : (t > 4294967295.0 ? 4294967295.0 : t)) : 0u;
  *keep_scale = (float)(1.0 / (1.0 - p));
  return true;
}

extern "C" int etpgt_gemm_bf16x3_gelu(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, int64_t M,
                                      int64_t N, int64_t K, int64_t lda, int64_t ldb, const float* bias, float* C,
                                      int64_t ldc, void* h_hi, void* h_lo, int64_t ldh, double drop_p, uint64_t seed,
                                      void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  ETPGT_REQUIRE(h_hi != nullptr && h_lo != nullptr && ldh >= N && ldh % 8 == 0 && N % 8 == 0,
                "gemm_bf16x3_gelu: h_hi / h_lo required, N and ldh multiples of 8, ldh >= N");
  ETPGT_REQUIRE((((uintptr_t)h_hi | (uintptr_t)h_lo) & 15) == 0, "gemm_bf16x3_gelu: outputs must be 16-byte aligned");
  ActEpilogue act = {};
  act.hi = static_cast<__nv_bfloat16*>(h_hi);
  act.lo = static_cast<__nv_bfloat16*>(h_lo);
  act.ld = ldh;
  act.seed = seed;
  ETPGT_REQUIRE(gelu_dropout_params(drop_p, &act.drop_threshold, &act.keep_scale),
                "gemm_bf16x3_gelu: dropout p must be in [0, 1)");
  return gemm_run(a_hi, a_lo, b_hi, b_lo, M, N, K, lda, ldb, 0, 0, bias, 0, C, ldc, 1, ws, ws_bytes, stream, act);
}

extern "C" int etpgt_gelu_bwd_split(const float* d_h, const float* u, int64_t rows, int64_t cols, double drop_p,
                                    uint64_t seed, void* hi, void* lo, int64_t ld_out, float* colsum, void* ws,
                                    size_t ws_bytes, etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  ETPGT_REQUIRE(rows >= 0 && cols > 0 && cols % 4 == 0 && ld_out >= cols, "gelu_bwd_split: bad sizes");
  ETPGT_REQUIRE(d_h != nullptr && u != nullptr && hi != nullptr && lo != nullptr, "gelu_bwd_split: null argument");
  uint32_t threshold;
  float keep_scale;
  ETPGT_REQUIRE(gelu_dropout_params(drop_p, &threshold, &keep_scale), "gelu_bwd_split: dropout p must be in [0, 1)");
  if (colsum != nullptr && ws_bytes < etpgt_split_bf16_workspace_bytes(rows, cols)) {
    set_error("gelu_bwd_split: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  const int64_t row_tiles = (rows + SPLIT_TILE - 1) / SPLIT_TILE, col_tiles = (cols + SPLIT_TILE - 1) / SPLIT_TILE;
  float* partial = colsum != nullptr ? static_cast<float*>(ws) : nullptr;
  if (rows > 0) {
    gelu_bwd_split_kernel<<<dim3((unsigned)col_tiles, (unsigned)row_tiles), 256, 0, stream>>>(
        d_h, u, rows, cols, seed, threshold, keep_scale, static_cast<__nv_bfloat16*>(hi),
        static_cast<__nv_bfloat16*>(lo), ld_out, partial);
    ETPGT_CHECK_LAUNCH("gelu_bwd_split");
  }
  if (colsum != nullptr) {
    colsum_reduce_kernel<<<(unsigned)((cols * 32 + 255) / 256), 256, 0, stream>>>(partial, rows > 0 ? row_tiles : 0, cols,
                                                                                 colsum);
    ETPGT_CHECK_LAUNCH("colsum_reduce");
  }
  return ETPGT_OK;
}

extern "C" int etpgt_gemm_bf16x3(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo, int64_t M,
                                 int64_t N, int64_t K, int64_t lda, int64_t ldb, const float* bias, float* C,
                                 int64_t ldc, int split_k, void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  return etpgt_gemm_bf16x3_ex(a_hi, a_lo, b_hi, b_lo, M, N, K, lda, ldb, 0, 0, bias, 0, C, ldc, split_k, ws, ws_bytes,
                              stream);
}
