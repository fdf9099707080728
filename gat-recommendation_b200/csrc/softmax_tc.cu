// Full-catalogue softmax cross-entropy on the tensor cores (sm_100a: tcgen05 + TMA), forward and backward.
//
// For session rows S [B, D], the item table E [I, D] (row padding_idx left out), targets t and temperature T:
//   z = S E^T / T,  lse = logsumexp_j z[:, j],  loss = sum_b (lse[b] - z[b, t[b]]) / B_total
//   G = (softmax(z) - onehot(t)) / (T B_total),  dS = G E,  dE += G^T S
// The [B, I] logits never exist in memory, not even in chunks.  One warp-specialised kernel serves all three
// passes.  A CTA keeps 128 "rows" of one operand on the TMEM lanes and streams 128-row tiles of the other operand
// (the "columns") through a TMA ring, one 64-wide k-block of hi / lo bf16 parts at a time:
//   FWD  rows = sessions, columns = items.  The epilogue folds each logits tile into a per-row online
//        (max, sum exp) and picks up the target's logit; a combine kernel merges the column ranges in order.
//   DS   rows = sessions, columns = items.  The epilogue turns the recomputed logits tile into G (fp32), splits it
//        into a bf16 pair in swizzled shared memory (K-major A operand), and the MMA warp adds G . E_tile into a
//        [128, D] TMEM accumulator.  The item tile is streamed a second time for that product: the same 128-row x
//        64-column TMA box that is the K-major B operand of the logits is the MN-major B operand of G . E_tile.
//   DE   the same with the roles swapped: rows = items, columns = sessions, lse and targets are per column.
// Every product is split-bf16 ("bf16x3": hi.hi + hi.lo + lo.hi, fp32 accumulation in TMEM), the convention of
// gemm_tc.cu.  TMEM: two 128-column logits buffers (the epilogue drains one while the next is computed) and, for
// the gradients, D accumulator columns.  Column ranges split across CTAs are combined in a fixed order: no
// atomics, bit-reproducible.
// The backward recomputes the forward's logits bit for bit (same MMA sequence, operands swapped in DE) and keeps
// them, lse and the running maxima in natural units (exp(x) = 2^(x log2 e) on the MUFU unit): where the softmax
// is exact — one eligible column, P = 1 — the gradient is exactly zero, not rounding noise.
// With PREC = ETPGT_SOFTMAX_BF16 (opt-in, a different numerical contract) S, the columns and G are rounded once to
// bf16 and every product is one MMA per k-step; the CTA's 128 rows x D then stay resident in shared memory (<= 64 KB)
// and the column tiles stream through a ring of single boxes.  Everything else is the same code.
//
// The same kernel, instantiated with POOL, computes the sampled softmax over one pool of M negatives shared by the
// batch, with the log-Q correction (Bengio & Senecal 2008; Jean et al. 2015; Yi et al. 2019).  For pool ids p [M]
// (ascending) and log_q[j] = log(M q(p_j)):
//   z_pos[b]  = s_b . e_{t_b} / T                  (the positive: no correction)
//   z[b, j]   = s_b . e_{p_j} / T - log_q[j]       (-inf where p_j == t_b or p_j == padding_idx)
//   lse[b]    = logsumexp(z_pos[b], z[b, :]),   loss = sum_b (lse[b] - z_pos[b]) / B_total
// exp(z_pos) + sum_j exp(z_j) is an unbiased estimate of the full partition function, and a pool holding every
// non-padding item once with log_q = 0 gives the full-catalogue loss.  The columns are the gathered pool rows; the
// accidental hits of a session are one range of positions of the sorted pool ([hit_lo, hit_hi), masked by a
// position compare) and the padding entries get log_q = +inf.  The positive is an fp32 gather-dot outside the
// kernel, folded into lse by the combine; DE writes d_pool [M, D] and two row scatters add it, and the
// positive's c_b s_b, into the table.
#include <math.h>

#include "tc_common.cuh"

namespace etpgt {
namespace {

using namespace tc;

constexpr int TILE = 128;                              // TMEM lanes = rows of a CTA = columns of a logits tile
constexpr int kThreads = 192;                          // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue
constexpr uint32_t KB_BYTES = TILE * BLOCK_K * 2;      // one 128-row x 64-k bf16 box: 16 KB
constexpr uint32_t STAGE_BYTES = 4 * KB_BYTES;         // row hi, row lo, column hi, column lo
constexpr uint32_t G_BYTES = 4 * KB_BYTES;             // G tile: hi then lo, two 64-column k-blocks each
constexpr uint32_t ACC_COL = 2 * TILE;                 // first TMEM column of the gradient accumulator
// The tensor cores add each MMA's products into the fp32 accumulator with truncation, not round-to-nearest: over a
// whole column range (thousands of MMAs) that bias reached 3e-4 relative in dS at 32,768 x 82,174.  The accumulator
// is therefore drained every kDrainTiles column tiles (192 MMAs) and summed in fp32 by the epilogue threads.
constexpr int kDrainTiles = 8;
constexpr float kLog2e = 1.4426950408889634f;

enum Mode { FWD = 0, DS = 1, DE = 2 };

// 2^x on the MUFU unit (relative error ~2^-22, far inside the 1e-4 bound; -inf -> 0)
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// position of `id` inside the 32 columns from `base` on, or -1: the per-element tests of a chunk become
// compares against a compile-time column index
__device__ __forceinline__ int chunk_pos(int64_t id, int64_t base) {
  const int64_t d = id - base;
  return d >= 0 && d < 32 ? (int)d : -1;
}
// one set of barriers for up to S ring stages; rfull (bf16 only) follows tmem_base so that the split-bf16 kernels keep
// their offsets
template <int S> struct __align__(8) Bars {
  uint64_t full[S], empty[S];
  uint64_t lfull[2], lempty[2];   // logits buffers
  uint64_t gfull, gempty;         // G tile in shared memory
  uint64_t accfull, accempty;    // gradient accumulator: one phase per drain group
  uint32_t tmem_base;
  uint64_t rfull;                 // bf16: the resident row tile
};

// Shared memory, in order: the resident row tile (bf16 only), the TMA ring, the G tile (DS, DE) and the barriers.
// split-bf16: ring stages of row hi, row lo, column hi, column lo (64 KB), G as hi and lo (64 KB).
// bf16: the CTA's 128 rows x D stay resident (<= 64 KB), the column tiles stream through a ring of single 16 KB boxes,
// and G is one bf16 copy (32 KB): 192 KB + 32 KB in DS / DE, one CTA per SM.
template <int MODE, int PREC = ETPGT_SOFTMAX_BF16X3> struct Cfg {
  static constexpr bool bf16 = PREC == ETPGT_SOFTMAX_BF16;
  static constexpr int stages = bf16 ? 8 : MODE == FWD ? 3 : 2;
  static constexpr uint32_t stage_bytes = bf16 ? KB_BYTES : STAGE_BYTES;
  static constexpr uint32_t rows_bytes = bf16 ? 4 * KB_BYTES : 0;
  static constexpr uint32_t g_bytes = MODE == FWD ? 0 : bf16 ? 2 * KB_BYTES : G_BYTES;
  static constexpr uint32_t tmem_cols = MODE == FWD ? 256 : 512;
  using Barriers = Bars<bf16 ? stages : 3>;
  static constexpr size_t smem = 1024 + rows_bytes + (size_t)stages * stage_bytes + g_bytes + 256;
};

struct Params {
  int64_t rows, cols;           // the logits of a CTA are rows x (its range of) cols
  int dim;
  int tiles_per_range, ranges;
  float inv_t;                  // 1 / T
  float gscale;                 // 1 / (T * B_total)
  const int64_t* targets;       // per row (FWD, DS) or per column (DE)
  const float* lse;             // natural log; per row (DS) or per column (DE)
  const float* d_loss;
  int64_t padding_idx;          // item id left out (-1: none)
  float* part;                  // FWD: [3][ranges][rows]; DS / DE with ranges > 1: [ranges][rows][dim]
  float* out;                   // DS: d_sess (written), DE: d_table (added), when ranges == 1
  const float* bias;            // POOL: per column (FWD, DS) or row (DE): log_q, +inf for a padding entry
  const int2* hits;             // POOL: per session, the pool positions [x, y) equal to its target
};

template <int MODE, bool POOL = false, int PREC = ETPGT_SOFTMAX_BF16X3>
__global__ void __launch_bounds__(kThreads, 1)
full_softmax_tc_kernel(const __grid_constant__ CUtensorMap map_r_hi, const __grid_constant__ CUtensorMap map_r_lo,
                       const __grid_constant__ CUtensorMap map_c_hi, const __grid_constant__ CUtensorMap map_c_lo,
                       const Params p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  using C = Cfg<MODE, PREC>;
  constexpr bool kBf16 = C::bf16;
  constexpr int kStages = C::stages;
  uint8_t* ring = smem + C::rows_bytes;  // bf16: the resident row tile comes first
  uint8_t* smem_g = ring + kStages * C::stage_bytes;
  auto* bars = reinterpret_cast<typename C::Barriers*>(smem_g + C::g_bytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int row_tiles = (int)((p.rows + TILE - 1) / TILE);
  const int col_tiles = (int)((p.cols + TILE - 1) / TILE);
  // consecutive CTAs take different row tiles of the same column range: they stream the same column tiles
  const int rt = blockIdx.x % row_tiles, range = blockIdx.x / row_tiles;
  const int ct0 = range * p.tiles_per_range;
  const int ct1 = min(ct0 + p.tiles_per_range, col_tiles);
  const int n = ct1 - ct0;
  const int nkb = p.dim / BLOCK_K;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&bars->lfull[b], 1); mbar_init(&bars->lempty[b], 4); }
    mbar_init(&bars->gfull, 4);
    mbar_init(&bars->gempty, 1);
    mbar_init(&bars->accfull, 1);
    mbar_init(&bars->accempty, 4);
    if constexpr (kBf16) mbar_init(&bars->rfull, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_r_hi);
    if constexpr (!kBf16) tma_prefetch_desc(&map_r_lo);
    tma_prefetch_desc(&map_c_hi);
    if constexpr (!kBf16) tma_prefetch_desc(&map_c_lo);
  }
  if (warp == 1) tmem_alloc(&bars->tmem_base, C::tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    if (kBf16 && lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      // the CTA's rows once, then the k-blocks of the column tiles one box per stage, in the order the MMA warp
      // consumes them: logits of tile j, then the gradient product of tile j - 1
      mbar_expect_tx(&bars->rfull, (uint32_t)nkb * KB_BYTES);
      for (int kb = 0; kb < nkb; ++kb)
        tma_load_2d(&map_r_hi, &bars->rfull, smem + kb * KB_BYTES, kb * BLOCK_K, rt * TILE);
      auto load = [&](int ct) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          mbar_expect_tx(&bars->full[stage], KB_BYTES);
          tma_load_2d(&map_c_hi, &bars->full[stage], ring + stage * KB_BYTES, kb * BLOCK_K, ct * TILE);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      };
      for (int j = 0; j < n; ++j) {
        load(ct0 + j);
        if (MODE != FWD && j > 0) load(ct0 + j - 1);
      }
      if (MODE != FWD) load(ct1 - 1);
    } else if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      // the k-blocks of column tile ct, with the row tile's (logits) or alone (second pass of the gradients)
      auto load = [&](int ct, bool with_rows) {
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* st = smem + stage * STAGE_BYTES;
          mbar_expect_tx(&bars->full[stage], with_rows ? STAGE_BYTES : 2 * KB_BYTES);
          if (with_rows) {
            tma_load_2d(&map_r_hi, &bars->full[stage], st, kb * BLOCK_K, rt * TILE);
            tma_load_2d(&map_r_lo, &bars->full[stage], st + KB_BYTES, kb * BLOCK_K, rt * TILE);
          }
          tma_load_2d(&map_c_hi, &bars->full[stage], st + 2 * KB_BYTES, kb * BLOCK_K, ct * TILE);
          tma_load_2d(&map_c_lo, &bars->full[stage], st + 3 * KB_BYTES, kb * BLOCK_K, ct * TILE);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      };
      // the order the MMA warp consumes: logits of tile j, then the gradient product of tile j - 1
      for (int j = 0; j < n; ++j) {
        load(ct0 + j, true);
        if (MODE != FWD && j > 0) load(ct0 + j - 1, false);
      }
      if (MODE != FWD) load(ct1 - 1, false);
    }
  } else if (warp == 1) {
    if (kBf16 && lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      constexpr uint32_t idesc_l = instr_desc_bf16(TILE, TILE);
      constexpr uint32_t idesc_g = instr_desc_bf16_major(TILE, BLOCK_K, false, true);
      const uint32_t rows = smem_u32(smem), g = smem_u32(smem_g);
      // the same gradient product as below with one bf16 G and one bf16 column tile: one MMA per k-step
      auto grad = [&](int j) {
        const int group = j / kDrainTiles;
        const bool group_start = j % kDrainTiles == 0, group_end = (j + 1) % kDrainTiles == 0 || j == n - 1;
        if (group_start && group > 0) mbar_wait(&bars->accempty, (uint32_t)(group - 1) & 1);  // drained
        mbar_wait(&bars->gfull, (uint32_t)j & 1);
        tc_fence_after();
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after();
          const uint32_t c = smem_u32(ring + stage * KB_BYTES);
          const uint32_t tmem_d = tmem_base + ACC_COL + (uint32_t)(kb * BLOCK_K);
#pragma unroll
          for (int kk = 0; kk < TILE / UMMA_K; ++kk) {
            const uint32_t off_a = (uint32_t)(kk >> 2) * KB_BYTES + (uint32_t)(kk & 3) * UMMA_K * 2;
            const uint32_t off_b = (uint32_t)kk * UMMA_K * 128;
            umma_bf16(tmem_d, make_desc_sw128(g + off_a), make_desc_mn_sw128(c + off_b, KB_BYTES), idesc_g,
                      (group_start && kk == 0) ? 0u : 1u);
          }
          umma_commit(&bars->empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bars->gempty);
        if (group_end) umma_commit(&bars->accfull);
      };
      mbar_wait(&bars->rfull, 0);
      tc_fence_after();
      for (int j = 0; j < n; ++j) {
        const int b = j & 1;
        mbar_wait(&bars->lempty[b], ((uint32_t)(j >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(b * TILE);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after();
          const uint32_t r = rows + (uint32_t)kb * KB_BYTES, c = smem_u32(ring + stage * KB_BYTES);
          // one product per k-step in the same k order in every pass (DE has the operands swapped), so the
          // recomputed logits are the forward's bit for bit
#pragma unroll
          for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
            const uint32_t off = (uint32_t)kk * UMMA_K * 2;
            umma_bf16(tmem_d, make_desc_sw128(r + off), make_desc_sw128(c + off), idesc_l,
                      (kb == 0 && kk == 0) ? 0u : 1u);
          }
          umma_commit(&bars->empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bars->lfull[b]);
        if (MODE != FWD && j > 0) grad(j - 1);
      }
      if (MODE != FWD) grad(n - 1);
    } else if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      constexpr uint32_t idesc_l = instr_desc_bf16(TILE, TILE);
      // G [rows, 128 columns] (K-major) x column tile [128 columns, 64 of D] (MN-major): one 64-wide slice of D
      constexpr uint32_t idesc_g = instr_desc_bf16_major(TILE, BLOCK_K, false, true);
      const uint32_t g_hi = smem_u32(smem_g), g_lo = g_hi + 2 * KB_BYTES;
      auto grad = [&](int j) {
        const int group = j / kDrainTiles;
        const bool group_start = j % kDrainTiles == 0, group_end = (j + 1) % kDrainTiles == 0 || j == n - 1;
        if (group_start && group > 0) mbar_wait(&bars->accempty, (uint32_t)(group - 1) & 1);  // drained
        mbar_wait(&bars->gfull, (uint32_t)j & 1);
        tc_fence_after();
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after();
          const uint32_t c_hi = smem_u32(smem + stage * STAGE_BYTES) + 2 * KB_BYTES, c_lo = c_hi + KB_BYTES;
          const uint32_t tmem_d = tmem_base + ACC_COL + (uint32_t)(kb * BLOCK_K);
#pragma unroll
          for (int kk = 0; kk < TILE / UMMA_K; ++kk) {
            // A: 32 bytes along a swizzle row of G's k-block kk / 4; B: 16 rows (2 KB) of the column tile
            const uint32_t off_a = (uint32_t)(kk >> 2) * KB_BYTES + (uint32_t)(kk & 3) * UMMA_K * 2;
            const uint32_t off_b = (uint32_t)kk * UMMA_K * 128;
            const uint32_t accumulate = (group_start && kk == 0) ? 0u : 1u;
            const uint64_t da_hi = make_desc_sw128(g_hi + off_a), da_lo = make_desc_sw128(g_lo + off_a);
            const uint64_t db_hi = make_desc_mn_sw128(c_hi + off_b, KB_BYTES);
            const uint64_t db_lo = make_desc_mn_sw128(c_lo + off_b, KB_BYTES);
            umma_bf16(tmem_d, da_hi, db_hi, idesc_g, accumulate);
            umma_bf16(tmem_d, da_hi, db_lo, idesc_g, 1u);
            umma_bf16(tmem_d, da_lo, db_hi, idesc_g, 1u);
          }
          umma_commit(&bars->empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bars->gempty);
        if (group_end) umma_commit(&bars->accfull);
      };
      for (int j = 0; j < n; ++j) {
        const int b = j & 1;
        mbar_wait(&bars->lempty[b], ((uint32_t)(j >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(b * TILE);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after();
          const uint32_t r_hi = smem_u32(smem + stage * STAGE_BYTES), r_lo = r_hi + KB_BYTES;
          const uint32_t c_hi = r_hi + 2 * KB_BYTES, c_lo = r_hi + 3 * KB_BYTES;
#pragma unroll
          for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
            const uint32_t off = (uint32_t)kk * UMMA_K * 2;
            const uint32_t accumulate = (kb == 0 && kk == 0) ? 0u : 1u;
            const uint64_t da_hi = make_desc_sw128(r_hi + off), db_hi = make_desc_sw128(c_hi + off);
            umma_bf16(tmem_d, da_hi, db_hi, idesc_l, accumulate);
            // the same three products in the same order in every pass (DE has the operands swapped), so the
            // recomputed logits are the forward's bit for bit
            if constexpr (MODE == DE) {
              umma_bf16(tmem_d, make_desc_sw128(r_lo + off), db_hi, idesc_l, 1u);
              umma_bf16(tmem_d, da_hi, make_desc_sw128(c_lo + off), idesc_l, 1u);
            } else {
              umma_bf16(tmem_d, da_hi, make_desc_sw128(c_lo + off), idesc_l, 1u);
              umma_bf16(tmem_d, make_desc_sw128(r_lo + off), db_hi, idesc_l, 1u);
            }
          }
          umma_commit(&bars->empty[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bars->lfull[b]);
        if (MODE != FWD && j > 0) grad(j - 1);
      }
      if (MODE != FWD) grad(n - 1);
    }
  } else {
    // TMEM lane quarter = warp % 4; thread = one row of the CTA
    const int q = warp & 3;
    const int r_local = q * 32 + lane;
    const int64_t row = (int64_t)rt * TILE + r_local;
    const bool row_ok = row < p.rows;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
    if constexpr (MODE == FWD) {
      const int64_t tgt = !POOL && row_ok ? p.targets[row] : -1;
      const int2 hit = POOL && row_ok ? p.hits[row] : make_int2(0, 0);
      float m = -INFINITY, s = 0.f, zt = 0.f;
      for (int j = 0; j < n; ++j) {
        const int b = j & 1;
        mbar_wait(&bars->lfull[b], (uint32_t)(j >> 1) & 1);
        tc_fence_after();
        const int64_t col0 = (int64_t)(ct0 + j) * TILE;
#pragma unroll 1
        for (int c = 0; c < TILE; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(lane_addr + (uint32_t)(b * TILE + c), v);
          if (c + 32 == TILE) {  // logits buffer fully read: the MMA warp may overwrite it
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->lempty[b]);
          }
          const int64_t base = col0 + c;
          const int lim = p.cols - base < 32 ? (int)(p.cols - base) : 32;
          float y[32];
          float mc = -INFINITY;
          if constexpr (POOL) {
            // lane e holds column e's log_q; the row's accidental hits as positions in the chunk
            const float bias_lane = lane < lim ? p.bias[base + lane] : 0.f;
            const int hit_lo = (int)max((int64_t)0, min((int64_t)32, hit.x - base));
            const int hit_hi = (int)max((int64_t)0, min((int64_t)32, hit.y - base));
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              y[e] = __fmaf_rn(__uint_as_float(v[e]), p.inv_t, -__shfl_sync(0xffffffffu, bias_lane, e));
              if (e >= lim || (e >= hit_lo && e < hit_hi)) y[e] = -INFINITY;
              mc = fmaxf(mc, y[e]);
            }
          } else {
            const int pad_e = chunk_pos(p.padding_idx, base), tgt_e = chunk_pos(tgt, base);
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              y[e] = __uint_as_float(v[e]) * p.inv_t;
              if (e >= lim || e == pad_e) y[e] = -INFINITY;
              if (e == tgt_e) zt = y[e];
              mc = fmaxf(mc, y[e]);
            }
          }
          if (mc == -INFINITY) continue;  // nothing of this chunk takes part
          if (mc > m) {
            s *= fast_exp2((m - mc) * kLog2e);
            m = mc;
          }
#pragma unroll
          for (int e = 0; e < 32; ++e) s += fast_exp2((y[e] - m) * kLog2e);
        }
      }
      if (row_ok) {
        p.part[(int64_t)range * p.rows + row] = m;
        p.part[((int64_t)p.ranges + range) * p.rows + row] = s;
        p.part[((int64_t)2 * p.ranges + range) * p.rows + row] = zt;
      }
    } else {
      const float gscale = __ldg(p.d_loss) * p.gscale;
      float lse_row = 0.f;
      int64_t tgt_row = -1;
      int2 hit = make_int2(0, 0);
      if (MODE == DS && row_ok) {
        lse_row = p.lse[row];
        if constexpr (POOL) hit = p.hits[row];
        else tgt_row = p.targets[row];
      }
      const float bias_row = POOL && MODE == DE && row_ok ? p.bias[row] : 0.f;
      uint8_t* g_row = smem_g + r_local * 128;
      const bool direct = p.ranges == 1;
      // POOL: rows of DE are pool positions, and d_pool is written whole
      const bool store = row_ok && !(!POOL && MODE == DE && row == p.padding_idx);
      float* dst = direct ? p.out + row * p.dim : p.part + ((int64_t)range * p.rows + row) * p.dim;
      // group `group` of column tiles is complete in the accumulator: add it to this thread's row in fp32 (the first
      // group overwrites, except that d_table is always accumulated into), then hand the accumulator back
      auto drain = [&](int group) {
        mbar_wait(&bars->accfull, (uint32_t)group & 1);
        tc_fence_after();
        const bool add = group > 0 || (!POOL && MODE == DE && direct);
#pragma unroll 1
        for (int c = 0; c < p.dim; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(lane_addr + ACC_COL + (uint32_t)c, v);
          if (c + 32 == p.dim) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->accempty);
          }
          if (!store) continue;
#pragma unroll
          for (int e = 0; e < 32; e += 4) {
            float4 o = make_float4(__uint_as_float(v[e]), __uint_as_float(v[e + 1]), __uint_as_float(v[e + 2]),
                                   __uint_as_float(v[e + 3]));
            if (add) o = add4(ld4(dst + c + e), o);
            st4(dst + c + e, o);
          }
        }
      };
      for (int j = 0; j < n; ++j) {
        const int b = j & 1;
        mbar_wait(&bars->lfull[b], (uint32_t)(j >> 1) & 1);
        mbar_wait(&bars->gempty, ((uint32_t)j & 1) ^ 1);  // the product of the previous G has completed
        tc_fence_after();
        const int64_t col0 = (int64_t)(ct0 + j) * TILE;
#pragma unroll 1
        for (int c = 0; c < TILE; c += 32) {
          uint32_t v[32];
          tmem_ld_32x32(lane_addr + (uint32_t)(b * TILE + c), v);
          if (c + 32 == TILE) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->lempty[b]);
          }
          const int64_t base = col0 + c;
          const int lim = !row_ok ? 0 : p.cols - base < 32 ? (int)(p.cols - base) : 32;
          // DS: the padding column and the row's target as positions in the chunk.  DE: the chunk's 32 columns are
          // sessions; lane e fetches column e's lse and its target as a row of this CTA (-1: none), shared by shuffles
          // POOL, DS: lane e holds column e's log_q, and the row's hits are positions in the chunk.  POOL, DE: lane e
          // packs session e's hits as rows of this CTA, [tgt_lane & 0xffff, tgt_lane >> 16)
          int pad_e = -1, tgt_e = -1, tgt_lane = POOL ? 0 : -1, hit_lo = 0, hit_hi = 0;
          float lse_lane = 0.f, bias_lane = 0.f;
          if constexpr (MODE == DS) {
            if constexpr (POOL) {
              if (base + lane < p.cols) bias_lane = p.bias[base + lane];
              hit_lo = (int)max((int64_t)0, min((int64_t)32, hit.x - base));
              hit_hi = (int)max((int64_t)0, min((int64_t)32, hit.y - base));
            } else {
              pad_e = chunk_pos(p.padding_idx, base);
              tgt_e = chunk_pos(tgt_row, base);
            }
          } else if (base + lane < p.cols) {
            lse_lane = p.lse[base + lane];
            if constexpr (POOL) {
              const int2 h = p.hits[base + lane];
              const int64_t r0 = (int64_t)rt * TILE;
              const int lo = (int)max((int64_t)0, min((int64_t)TILE, h.x - r0));
              const int hi = (int)max((int64_t)0, min((int64_t)TILE, h.y - r0));
              tgt_lane = lo | (hi << 16);
            } else {
              const int64_t t = p.targets[base + lane] - (int64_t)rt * TILE;
              tgt_lane = t >= 0 && t < TILE ? (int)t : -1;
            }
          }
          float g[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            const float y = __uint_as_float(v[e]) * p.inv_t;
            float pr;
            if constexpr (POOL && MODE == DS) {
              const float z = __fmaf_rn(__uint_as_float(v[e]), p.inv_t, -__shfl_sync(0xffffffffu, bias_lane, e));
              pr = fast_exp2((z - lse_row) * kLog2e);
              if (e >= lim || (e >= hit_lo && e < hit_hi)) pr = 0.f;
            } else if constexpr (POOL) {
              const float l = __shfl_sync(0xffffffffu, lse_lane, e);
              const int t = __shfl_sync(0xffffffffu, tgt_lane, e);
              const float z = __fmaf_rn(__uint_as_float(v[e]), p.inv_t, -bias_row);
              pr = fast_exp2((z - l) * kLog2e);
              if (e >= lim || (r_local >= (t & 0xffff) && r_local < (t >> 16))) pr = 0.f;
            } else if constexpr (MODE == DS) {
              pr = fast_exp2((y - lse_row) * kLog2e) - (e == tgt_e ? 1.f : 0.f);
              if (e >= lim || e == pad_e) pr = 0.f;
            } else {
              const float l = __shfl_sync(0xffffffffu, lse_lane, e);
              const int t = __shfl_sync(0xffffffffu, tgt_lane, e);
              pr = fast_exp2((y - l) * kLog2e) - (t == r_local ? 1.f : 0.f);
              if (e >= lim) pr = 0.f;
            }
            g[e] = pr * gscale;
          }
          // split into the bf16 pair (bf16: only hi is stored, G rounded once); 128-byte swizzle of the K-major A
          // operand (16-byte unit ^ row % 8)
          uint8_t* g_kb = g_row + (c >> 6) * KB_BYTES;
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            uint32_t h[4], l[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const float x0 = g[8 * u + 2 * t], x1 = g[8 * u + 2 * t + 1];
              const __nv_bfloat16 h0 = __float2bfloat16_rn(x0), h1 = __float2bfloat16_rn(x1);
              const __nv_bfloat16 l0 = __float2bfloat16_rn(x0 - __bfloat162float(h0));
              const __nv_bfloat16 l1 = __float2bfloat16_rn(x1 - __bfloat162float(h1));
              h[t] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
              l[t] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
            }
            const uint32_t off = (uint32_t)(((((c & 63) >> 3) + u) ^ (lane & 7)) << 4);
            *reinterpret_cast<uint4*>(g_kb + off) = make_uint4(h[0], h[1], h[2], h[3]);
            if constexpr (!kBf16)
              *reinterpret_cast<uint4*>(g_kb + 2 * KB_BYTES + off) = make_uint4(l[0], l[1], l[2], l[3]);
          }
        }
        fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor cores
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->gfull);
        if ((j + 1) % kDrainTiles == 0 || j == n - 1) drain(j / kDrainTiles);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::tmem_cols);
  }
}

// lse[b] and the loss from the per-range (max, sum) partials, ranges merged in ascending order, rows summed by a
// fixed tree: one block, deterministic.
constexpr int kCombineThreads = 1024;
__global__ void __launch_bounds__(kCombineThreads)
fwd_combine_kernel(const float* __restrict__ part, int ranges, int tiles_per_range, int64_t rows, int64_t cols,
                   const int64_t* __restrict__ targets, double total, float* __restrict__ lse, float* __restrict__ loss) {
  __shared__ double red[kCombineThreads];
  double acc = 0.0;
  for (int64_t b = threadIdx.x; b < rows; b += kCombineThreads) {
    float m = -INFINITY;
    for (int r = 0; r < ranges; ++r) m = fmaxf(m, part[(int64_t)r * rows + b]);
    float s = 0.f;
    for (int r = 0; r < ranges; ++r) {
      const float mr = part[(int64_t)r * rows + b];
      if (mr != -INFINITY) s += part[((int64_t)ranges + r) * rows + b] * exp2f((mr - m) * kLog2e);
    }
    const float l = m + logf(s);
    const int64_t t = targets[b];
    const float zt = (t >= 0 && t < cols) ? part[((int64_t)2 * ranges + (t / TILE) / tiles_per_range) * rows + b] : 0.f;
    lse[b] = l;
    acc += (double)(l - zt);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int w = kCombineThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = (float)(red[0] / total);
}

// out[row] (=|+=) sum_r part[r][row], r ascending; DE leaves row padding_idx untouched
__global__ void __launch_bounds__(256)
grad_combine_kernel(const float* __restrict__ part, int ranges, int64_t rows, int dim, int accumulate,
                    int64_t skip_row, float* __restrict__ out) {
  const int64_t total4 = rows * dim / 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
    if ((4 * i) / dim == skip_row) continue;
    float4 acc = accumulate ? ld4(out + 4 * i) : zero4();
    for (int r = 0; r < ranges; ++r) acc = add4(acc, ldg4(part + (int64_t)r * rows * dim + 4 * i));
    st4(out + 4 * i, acc);
  }
}

struct Plan {
  int tiles_per_range, ranges, grid;
};

// Column ranges per row tile: the count that minimises (waves of CTAs) x (column tiles per CTA), the fewest on a
// tie, at most max_ranges.
Plan plan_ranges(int64_t rows, int64_t cols, int max_ranges) {
  const int64_t row_tiles = (rows + TILE - 1) / TILE, col_tiles = (cols + TILE - 1) / TILE;
  int64_t best_cost = -1;
  Plan best = {};
  const int64_t top = col_tiles < max_ranges ? col_tiles : max_ranges;
  for (int64_t want = 1; want <= top; ++want) {
    const int64_t tpr = (col_tiles + want - 1) / want, r = (col_tiles + tpr - 1) / tpr;
    const int64_t cost = ((row_tiles * r + kNumSMs - 1) / kNumSMs) * tpr;
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best.tiles_per_range = (int)tpr;
      best.ranges = (int)r;
      best.grid = (int)(row_tiles * r);
    }
  }
  return best;
}
// forward partials are 3 floats per (row, range): ranges are limited by the column tiles only
Plan plan_fwd(int64_t batch, int64_t items) { return plan_ranges(batch, items, 1 << 20); }
// gradient partials are [ranges][rows][D]: at most about four waves' worth of CTAs, so the workspace stays
// within a few row-tile multiples of B x D (I x D)
Plan plan_grad(int64_t rows, int64_t cols) {
  const int64_t row_tiles = (rows + TILE - 1) / TILE;
  const int64_t cap = (4 * kNumSMs + row_tiles - 1) / row_tiles;
  return plan_ranges(rows, cols, (int)(cap < 1 ? 1 : cap));
}

bool softmax_dim_ok(int dim) { return dim == 64 || dim == 128 || dim == 192 || dim == 256; }

// The workspace of one call, in carve order: the bf16 pairs of the session rows and of the columns (the table, or
// the gathered pool), the partials (the forward's [3][ranges][B] or a split gradient pass's [ranges][rows][D],
// whichever is larger), then the pool loss's own buffers, which are 0 for the full loss.
struct Layout {
  size_t s_pair, c_pair, part, d_pool, bias, hits, coef, scatter;
  size_t total() const { return 2 * s_pair + 2 * c_pair + part + d_pool + bias + hits + coef + scatter + 256; }
};
Layout layout(int64_t batch, int64_t cols, int dim) {
  Layout l = {};
  l.s_pair = align_up((size_t)batch * dim * 2);
  l.c_pair = align_up((size_t)cols * dim * 2);
  const Plan pf = plan_fwd(batch, cols), ps = plan_grad(batch, cols), pe = plan_grad(cols, batch);
  const size_t fp = (size_t)3 * pf.ranges * batch * sizeof(float);
  const size_t gs = ps.ranges > 1 ? (size_t)ps.ranges * batch * dim * sizeof(float) : 0;
  const size_t ge = pe.ranges > 1 ? (size_t)pe.ranges * cols * dim * sizeof(float) : 0;
  const size_t g = gs > ge ? gs : ge;
  l.part = align_up(fp > g ? fp : g);
  return l;
}

// the tensor maps of the session and column pairs and the buffers carved for them; the pool's stay null for the
// full loss
struct Operands {
  CUtensorMap s_hi, s_lo, c_hi, c_lo;
  void* s_slots = nullptr;      // the session pair's 2 * s_pair bytes
  float* part = nullptr;
  float *d_pool = nullptr, *bias = nullptr, *coef = nullptr;
  int2* hits = nullptr;
  void* scatter_ws = nullptr;
  size_t scatter_bytes = 0;
};

// the checks of both losses, in this order: dim, the loss's own size ranges (`ranges()` sets the message and returns
// ETPGT_EINVAL when one fails), null arguments, temperature and padding_idx
template <class Ranges>
int check_args(const char* name, int dim, Ranges ranges, bool args_set, float temperature, int64_t padding_idx,
               int64_t items) {
  ETPGT_REQUIRE(softmax_dim_ok(dim), "%s: dim %d is not supported (dim must be one of 64, 128, 192, 256)", name, dim);
  const int rc = ranges();
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(args_set, "%s: null argument", name);
  ETPGT_REQUIRE(temperature > 0.f, "%s: temperature must be positive", name);
  ETPGT_REQUIRE(padding_idx >= -1 && padding_idx < items, "%s: padding_idx must be -1 or an item id", name);
  return ETPGT_OK;
}

// Checks the workspace, carves the two bf16 pairs and the partials, splits sess, lets `columns(w, c_hi, c_lo)` fill
// the column pair (and carve what else the loss needs from w), then encodes the four tensor maps.  bf16: the same
// carve, but sess and the columns are rounded once into the hi slots (c_lo is null for `columns`), the lo slots stay
// unused and the lo maps are the hi maps.
template <class Columns>
int prepare(const char* name, const Layout& l, const float* sess, int64_t batch, int64_t cols, int dim, bool bf16,
            void* ws, size_t ws_bytes, cudaStream_t stream, Operands* o, Columns columns) {
  if (ws == nullptr || ws_bytes < l.total()) {
    set_error("%s: workspace too small (%zu < %zu bytes)", name, ws_bytes, l.total());
    return ETPGT_EWORKSPACE;
  }
  Workspace w(ws, ws_bytes);
  void* s_hi = w.take<char>(l.s_pair);
  void* s_lo = w.take<char>(l.s_pair);
  auto* c_hi = w.take<__nv_bfloat16>(l.c_pair / 2);
  auto* c_lo = w.take<__nv_bfloat16>(l.c_pair / 2);
  o->part = w.take<float>(l.part / sizeof(float));
  o->s_slots = s_hi;
  int rc = bf16 ? etpgt_f32_to_bf16(sess, s_hi, batch * dim, stream)
                : etpgt_split_bf16(sess, batch, dim, dim, s_hi, s_lo, dim, nullptr, nullptr, 0, nullptr, nullptr, 0,
                                   stream);
  if (rc != ETPGT_OK) return rc;
  rc = columns(w, c_hi, bf16 ? nullptr : c_lo);
  if (rc != ETPGT_OK) return rc;
  if (!(make_map_bf16(&o->s_hi, s_hi, batch, dim, dim, TILE) && make_map_bf16(&o->c_hi, c_hi, cols, dim, dim, TILE) &&
        (bf16 || (make_map_bf16(&o->s_lo, s_lo, batch, dim, dim, TILE) &&
                  make_map_bf16(&o->c_lo, c_lo, cols, dim, dim, TILE))))) {
    set_error("%s: cuTensorMapEncodeTiled failed", name);
    return ETPGT_ECUDA;
  }
  if (bf16) {
    o->s_lo = o->s_hi;
    o->c_lo = o->c_hi;
  }
  return ETPGT_OK;
}

// precision is one of the two ETPGT_SOFTMAX_* values
int check_precision(const char* name, int precision) {
  ETPGT_REQUIRE(precision == ETPGT_SOFTMAX_BF16X3 || precision == ETPGT_SOFTMAX_BF16,
                "%s: precision %d is not supported (ETPGT_SOFTMAX_BF16X3 = 0 or ETPGT_SOFTMAX_BF16 = 1)", name,
                precision);
  return ETPGT_OK;
}

// the loss is the mean over total_sessions, or over the batch when that is not positive
double mean_over(double total_sessions, int64_t batch) { return total_sessions > 0 ? total_sessions : (double)batch; }

// the Params every pass of one call shares; each pass sets rows, cols, its column ranges and out
Params call_params(int dim, float temperature, double total, int64_t padding_idx, const Operands& o,
                   const int64_t* targets, const float* lse = nullptr, const float* d_loss = nullptr) {
  Params p = {};
  p.dim = dim;
  p.inv_t = 1.f / temperature;
  p.gscale = (float)(1.0 / ((double)temperature * total));
  p.targets = targets;
  p.lse = lse;
  p.d_loss = d_loss;
  p.padding_idx = padding_idx;
  p.part = o.part;
  p.bias = o.bias;
  p.hits = o.hits;
  return p;
}

template <int MODE, bool POOL, int PREC>
int launch_prec(const CUtensorMap& r_hi, const CUtensorMap& r_lo, const CUtensorMap& c_hi, const CUtensorMap& c_lo,
                const Params& p, int grid, const char* name, cudaStream_t stream) {
  using C = Cfg<MODE, PREC>;
  const size_t smem = C::smem + sizeof(typename C::Barriers);
  cudaFuncSetAttribute(full_softmax_tc_kernel<MODE, POOL, PREC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                       (int)smem);
  full_softmax_tc_kernel<MODE, POOL, PREC><<<grid, kThreads, smem, stream>>>(r_hi, r_lo, c_hi, c_lo, p);
  ETPGT_CHECK_LAUNCH(name);
  return ETPGT_OK;
}
// the kernel of `precision`; a bf16 call's lo maps are its hi maps and are not read
template <int MODE, bool POOL = false>
int launch(const CUtensorMap& r_hi, const CUtensorMap& r_lo, const CUtensorMap& c_hi, const CUtensorMap& c_lo,
           const Params& p, int grid, const char* name, int precision, cudaStream_t stream) {
  return precision == ETPGT_SOFTMAX_BF16
             ? launch_prec<MODE, POOL, ETPGT_SOFTMAX_BF16>(r_hi, r_lo, c_hi, c_lo, p, grid, name, stream)
             : launch_prec<MODE, POOL, ETPGT_SOFTMAX_BF16X3>(r_hi, r_lo, c_hi, c_lo, p, grid, name, stream);
}

// One gradient pass (DS or DE) over rows x cols into out [rows, D].  Split into column ranges, its partials are
// summed into out in range order (added to out when `accumulate`, row skip_row left alone).
template <int MODE, bool POOL = false>
int grad_pass(const CUtensorMap& r_hi, const CUtensorMap& r_lo, const CUtensorMap& c_hi, const CUtensorMap& c_lo,
              Params p, int64_t rows, int64_t cols, float* out, int accumulate, int64_t skip_row, const char* name,
              const char* combine_name, int precision, cudaStream_t stream) {
  const Plan pl = plan_grad(rows, cols);
  p.rows = rows;
  p.cols = cols;
  p.tiles_per_range = pl.tiles_per_range;
  p.ranges = pl.ranges;
  p.out = out;
  const int rc = launch<MODE, POOL>(r_hi, r_lo, c_hi, c_lo, p, pl.grid, name, precision, stream);
  if (rc != ETPGT_OK) return rc;
  if (pl.ranges > 1) {
    grad_combine_kernel<<<grid_for(rows * p.dim / 4, 256, 8), 256, 0, stream>>>(p.part, pl.ranges, rows, p.dim,
                                                                                accumulate, skip_row, out);
    ETPGT_CHECK_LAUNCH(combine_name);
  }
  return ETPGT_OK;
}

// ---------------------------------------------------------------------------- full-catalogue softmax: host

int full_check_args(const float* sess, const float* table, const int64_t* targets, int64_t batch, int64_t items,
                    int dim, float temperature, int64_t padding_idx) {
  const auto ranges = [&] {
    ETPGT_REQUIRE(batch >= 1 && items >= 2 && batch < (int64_t(1) << 31) && items < (int64_t(1) << 31),
                  "full_softmax: need batch >= 1 and num_items >= 2 (got %lld, %lld)", (long long)batch,
                  (long long)items);
    return ETPGT_OK;
  };
  return check_args("full_softmax", dim, ranges, sess != nullptr && table != nullptr && targets != nullptr,
                    temperature, padding_idx, items);
}

// the columns are the table, split into its bf16 pair (bf16: rounded once)
int full_prepare(const float* sess, const float* table, int64_t batch, int64_t items, int dim, bool bf16, void* ws,
                 size_t ws_bytes, cudaStream_t stream, Operands* o) {
  return prepare("full_softmax", layout(batch, items, dim), sess, batch, items, dim, bf16, ws, ws_bytes, stream, o,
                 [&](Workspace&, __nv_bfloat16* c_hi, __nv_bfloat16* c_lo) {
                   if (c_lo == nullptr) return etpgt_f32_to_bf16(table, c_hi, items * dim, stream);
                   return etpgt_split_bf16(table, items, dim, dim, c_hi, c_lo, dim, nullptr, nullptr, 0, nullptr,
                                           nullptr, 0, stream);
                 });
}

// ---------------------------------------------------------------------------- shared-pool softmax: small kernels

// pool rows gathered from the table and split into the bf16 pair (hi = bf16(x), lo = bf16(x - hi), as
// etpgt_split_bf16; hi only when lo is null), and bias[j] = log_q[j], or +inf for a padding entry (its logit is then
// -inf in every pass)
__global__ void __launch_bounds__(256)
pool_gather_split_kernel(const int64_t* __restrict__ pool, const float* __restrict__ log_q,
                         const float* __restrict__ table, int64_t m, int dim, int64_t padding_idx,
                         __nv_bfloat16* __restrict__ hi, __nv_bfloat16* __restrict__ lo, float* __restrict__ bias) {
  const int q = dim / 4;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < m * q; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / q;
    const int64_t id = pool[j];
    const int k = (int)(i - j * q) * 4;
    if (k == 0) bias[j] = id == padding_idx ? INFINITY : log_q[j];
    const float4 x = ldg4(table + id * dim + k);
    const float xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const __nv_bfloat16 h = __float2bfloat16_rn(xs[t]);
      hi[j * dim + k + t] = h;
      if (lo != nullptr) lo[j * dim + k + t] = __float2bfloat16_rn(xs[t] - __bfloat162float(h));
    }
  }
}

// x, or x rounded to bf16 (round to nearest even) and back: the operands of the bf16 loss
template <bool BF16>
__device__ __forceinline__ float operand(float x) {
  if constexpr (BF16) return __bfloat162float(__float2bfloat16_rn(x));
  return x;
}

// one warp per session: its hit range [lower_bound, upper_bound) of the target in the sorted pool and, with
// z_pos != NULL, z_pos = (s_b . e_{t_b}) / T in fp32 (lane-strided products, then a fixed butterfly; BF16: of the
// rounded operands, whose products are exact)
template <bool BF16 = false>
__global__ void __launch_bounds__(256)
pool_rows_kernel(const float* __restrict__ sess, const float* __restrict__ table, const int64_t* __restrict__ targets,
                 const int64_t* __restrict__ pool, int64_t batch, int64_t m, int dim, float inv_t,
                 int2* __restrict__ hits, float* __restrict__ z_pos) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t b = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); b < batch; b += nwarps) {
    const int64_t t = targets[b];
    if (lane == 0) {
      int64_t lo = 0, hi = m;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (pool[mid] < t) lo = mid + 1; else hi = mid;
      }
      int64_t lo2 = lo, hi2 = m;
      while (lo2 < hi2) {
        const int64_t mid = (lo2 + hi2) >> 1;
        if (pool[mid] <= t) lo2 = mid + 1; else hi2 = mid;
      }
      hits[b] = make_int2((int)lo, (int)lo2);
    }
    if (z_pos == nullptr) continue;
    float acc = 0.f;
    for (int k = lane; k < dim; k += 32)
      acc = fmaf(operand<BF16>(sess[b * dim + k]), operand<BF16>(table[t * dim + k]), acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) z_pos[b] = acc * inv_t;
  }
}

// lse[b] = logsumexp of the per-range (max, sum) partials and z_pos[b], ranges merged in ascending order; the loss
// sum_b (lse[b] - z_pos[b]) / total by a fixed tree: one block, deterministic
__global__ void __launch_bounds__(kCombineThreads)
pool_combine_kernel(const float* __restrict__ part, int ranges, int64_t rows, const float* __restrict__ z_pos,
                    double total, float* __restrict__ lse, float* __restrict__ loss) {
  __shared__ double red[kCombineThreads];
  double acc = 0.0;
  for (int64_t b = threadIdx.x; b < rows; b += kCombineThreads) {
    const float zp = z_pos[b];
    float m = zp;
    for (int r = 0; r < ranges; ++r) m = fmaxf(m, part[(int64_t)r * rows + b]);
    float s = exp2f((zp - m) * kLog2e);
    for (int r = 0; r < ranges; ++r) {
      const float mr = part[(int64_t)r * rows + b];
      if (mr != -INFINITY) s += part[((int64_t)ranges + r) * rows + b] * exp2f((mr - m) * kLog2e);
    }
    const float l = m + logf(s);
    lse[b] = l;
    acc += (double)(l - zp);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int w = kCombineThreads / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = (float)(red[0] / total);
}

// the positive's gradient: coef[b] = d_loss (exp(z_pos - lse) - 1) / (T B_total) and, with d_sess != NULL,
// d_sess[b] += coef[b] e_{t_b}; one warp per session.  BF16: coef[b] is the positive's entry of G, computed as the
// loss kernel computes G and rounded to bf16 like it, and d_sess[b] += coef[b] bf16(e_{t_b}) (an exact product)
template <bool BF16 = false>
__global__ void __launch_bounds__(256)
pool_positive_bwd_kernel(const float* __restrict__ table, const int64_t* __restrict__ targets,
                         const float* __restrict__ z_pos, const float* __restrict__ lse, const float* __restrict__ d_loss,
                         int64_t batch, int dim, float gscale, float* __restrict__ coef, float* __restrict__ d_sess) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const float dl = __ldg(d_loss) * gscale;
  for (int64_t b = blockIdx.x * (int64_t)(blockDim.x >> 5) + (threadIdx.x >> 5); b < batch; b += nwarps) {
    const float c = BF16 ? operand<true>((fast_exp2((z_pos[b] - lse[b]) * kLog2e) - 1.f) * dl)
                         : dl * (expf(z_pos[b] - lse[b]) - 1.f);
    if (lane == 0) coef[b] = c;
    if (d_sess == nullptr) continue;
    const float* e = table + targets[b] * dim;
    for (int k = lane; k < dim; k += 32) d_sess[b * dim + k] = fmaf(c, operand<BF16>(e[k]), d_sess[b * dim + k]);
  }
}

// dst = bf16(src) as fp32: the rounded sessions whose rows the bf16 loss's positive adds to the table
__global__ void __launch_bounds__(256) round_bf16_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                         int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = operand<true>(src[i]);
}

// ---------------------------------------------------------------------------- shared-pool softmax: host

// the full loss's layout over the M pool rows, plus d_pool, the pool's bias, the sessions' hit ranges and positive
// coefficients, and the workspace of the two row scatters
Layout pool_layout(int64_t batch, int64_t m, int dim) {
  Layout l = layout(batch, m, dim);
  l.d_pool = align_up((size_t)m * dim * sizeof(float));
  l.bias = align_up((size_t)m * sizeof(float));
  l.hits = align_up((size_t)batch * sizeof(int2));
  l.coef = align_up((size_t)batch * sizeof(float));
  l.scatter = align_up(etpgt_scatter_rows_workspace_bytes(batch > m ? batch : m));
  return l;
}

int pool_check_args(const float* sess, const float* table, const int64_t* targets, const int64_t* pool_ids,
                    const float* log_q, int64_t batch, int64_t items, int64_t m, int dim, float temperature,
                    int64_t padding_idx) {
  const auto ranges = [&] {
    ETPGT_REQUIRE(batch >= 1 && batch < (int64_t(1) << 31), "pool_softmax: batch must be in [1, 2^31) (got %lld)",
                  (long long)batch);
    ETPGT_REQUIRE(m >= 1 && m < (int64_t(1) << 31), "pool_softmax: num_sampled must be in [1, 2^31) (got %lld)",
                  (long long)m);
    ETPGT_REQUIRE(items >= 1 && items < (int64_t(1) << 31), "pool_softmax: num_items must be in [1, 2^31) (got %lld)",
                  (long long)items);
    return ETPGT_OK;
  };
  return check_args("pool_softmax", dim, ranges,
                    sess != nullptr && table != nullptr && targets != nullptr && pool_ids != nullptr && log_q != nullptr,
                    temperature, padding_idx, items);
}

// the columns are the pool rows, gathered and split (bf16: rounded once); also finds the hit ranges (and z_pos when
// given)
int pool_prepare(const float* sess, const float* table, const int64_t* targets, const int64_t* pool_ids,
                 const float* log_q, int64_t batch, int64_t m, int dim, float inv_t, int64_t padding_idx, bool bf16,
                 float* z_pos, void* ws, size_t ws_bytes, cudaStream_t stream, Operands* o) {
  const Layout l = pool_layout(batch, m, dim);
  return prepare("pool_softmax", l, sess, batch, m, dim, bf16, ws, ws_bytes, stream, o,
                 [&](Workspace& w, __nv_bfloat16* c_hi, __nv_bfloat16* c_lo) {
                   o->d_pool = w.take<float>(l.d_pool / sizeof(float));
                   o->bias = w.take<float>(l.bias / sizeof(float));
                   o->hits = w.take<int2>(l.hits / sizeof(int2));
                   o->coef = w.take<float>(l.coef / sizeof(float));
                   o->scatter_bytes = l.scatter;
                   o->scatter_ws = w.take<char>(l.scatter);
                   pool_gather_split_kernel<<<grid_for(m * dim / 4, 256, 8), 256, 0, stream>>>(
                       pool_ids, log_q, table, m, dim, padding_idx, c_hi, c_lo, o->bias);
                   ETPGT_CHECK_LAUNCH("pool_softmax_gather");
                   if (bf16)
                     pool_rows_kernel<true><<<grid_for(batch, 8, 8), 256, 0, stream>>>(
                         sess, table, targets, pool_ids, batch, m, dim, inv_t, o->hits, z_pos);
                   else
                     pool_rows_kernel<<<grid_for(batch, 8, 8), 256, 0, stream>>>(sess, table, targets, pool_ids, batch,
                                                                                 m, dim, inv_t, o->hits, z_pos);
                   ETPGT_CHECK_LAUNCH("pool_softmax_rows");
                   return ETPGT_OK;
                 });
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" size_t etpgt_full_softmax_workspace_bytes(int64_t batch, int64_t num_items, int dim) {
  if (batch < 1 || num_items < 1 || dim < 1) return 256;
  return layout(batch, num_items, dim).total();
}

extern "C" int etpgt_full_softmax_fwd_ex(const float* sess, const float* table, const int64_t* targets, int64_t batch,
                                         int64_t num_items, int dim, float temperature, double total_sessions,
                                         int64_t padding_idx, float* lse, float* loss, void* ws, size_t ws_bytes,
                                         etpgt_stream_t stream_, int precision) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_precision("full_softmax_fwd", precision);
  if (rc != ETPGT_OK) return rc;
  rc = full_check_args(sess, table, targets, batch, num_items, dim, temperature, padding_idx);
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(lse != nullptr && loss != nullptr, "full_softmax_fwd: lse and loss are required");
  Operands o;
  rc = full_prepare(sess, table, batch, num_items, dim, precision == ETPGT_SOFTMAX_BF16, ws, ws_bytes, stream, &o);
  if (rc != ETPGT_OK) return rc;
  const double total = mean_over(total_sessions, batch);
  const Plan pl = plan_fwd(batch, num_items);
  Params p = call_params(dim, temperature, total, padding_idx, o, targets);
  p.rows = batch;
  p.cols = num_items;
  p.tiles_per_range = pl.tiles_per_range;
  p.ranges = pl.ranges;
  rc = launch<FWD>(o.s_hi, o.s_lo, o.c_hi, o.c_lo, p, pl.grid, "full_softmax_fwd", precision, stream);
  if (rc != ETPGT_OK) return rc;
  fwd_combine_kernel<<<1, kCombineThreads, 0, stream>>>(o.part, pl.ranges, pl.tiles_per_range, batch, num_items,
                                                        targets, total, lse, loss);
  ETPGT_CHECK_LAUNCH("full_softmax_fwd_combine");
  return ETPGT_OK;
}

extern "C" int etpgt_full_softmax_fwd(const float* sess, const float* table, const int64_t* targets, int64_t batch,
                                      int64_t num_items, int dim, float temperature, double total_sessions,
                                      int64_t padding_idx, float* lse, float* loss, void* ws, size_t ws_bytes,
                                      etpgt_stream_t stream) {
  return etpgt_full_softmax_fwd_ex(sess, table, targets, batch, num_items, dim, temperature, total_sessions,
                                   padding_idx, lse, loss, ws, ws_bytes, stream, ETPGT_SOFTMAX_BF16X3);
}

extern "C" int etpgt_full_softmax_bwd_ex(const float* sess, const float* table, const int64_t* targets,
                                         const float* lse, const float* d_loss, int64_t batch, int64_t num_items,
                                         int dim, float temperature, double total_sessions, int64_t padding_idx,
                                         float* d_sess, float* d_table_accumulate, void* ws, size_t ws_bytes,
                                         etpgt_stream_t stream_, int precision) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_precision("full_softmax_bwd", precision);
  if (rc != ETPGT_OK) return rc;
  rc = full_check_args(sess, table, targets, batch, num_items, dim, temperature, padding_idx);
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(lse != nullptr && d_loss != nullptr, "full_softmax_bwd: lse and d_loss are required");
  if (d_sess == nullptr && d_table_accumulate == nullptr) return ETPGT_OK;
  Operands o;
  rc = full_prepare(sess, table, batch, num_items, dim, precision == ETPGT_SOFTMAX_BF16, ws, ws_bytes, stream, &o);
  if (rc != ETPGT_OK) return rc;
  const Params p =
      call_params(dim, temperature, mean_over(total_sessions, batch), padding_idx, o, targets, lse, d_loss);
  if (d_sess != nullptr) {
    rc = grad_pass<DS>(o.s_hi, o.s_lo, o.c_hi, o.c_lo, p, batch, num_items, d_sess, 0, -1, "full_softmax_bwd_sess",
                       "full_softmax_bwd_sess_combine", precision, stream);
    if (rc != ETPGT_OK) return rc;
  }
  if (d_table_accumulate != nullptr) {
    rc = grad_pass<DE>(o.c_hi, o.c_lo, o.s_hi, o.s_lo, p, num_items, batch, d_table_accumulate, 1, padding_idx,
                       "full_softmax_bwd_table", "full_softmax_bwd_table_combine", precision, stream);
    if (rc != ETPGT_OK) return rc;
  }
  return ETPGT_OK;
}

extern "C" int etpgt_full_softmax_bwd(const float* sess, const float* table, const int64_t* targets, const float* lse,
                                      const float* d_loss, int64_t batch, int64_t num_items, int dim, float temperature,
                                      double total_sessions, int64_t padding_idx, float* d_sess,
                                      float* d_table_accumulate, void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  return etpgt_full_softmax_bwd_ex(sess, table, targets, lse, d_loss, batch, num_items, dim, temperature,
                                   total_sessions, padding_idx, d_sess, d_table_accumulate, ws, ws_bytes, stream,
                                   ETPGT_SOFTMAX_BF16X3);
}

extern "C" size_t etpgt_pool_softmax_workspace_bytes(int64_t batch, int64_t num_sampled, int dim) {
  if (batch < 1 || num_sampled < 1 || dim < 1) return 256;
  return pool_layout(batch, num_sampled, dim).total();
}

extern "C" int etpgt_pool_softmax_fwd_ex(const float* sess, const float* table, const int64_t* targets,
                                         const int64_t* pool_ids, const float* log_q, int64_t batch,
                                         int64_t num_items, int64_t num_sampled, int dim, float temperature,
                                         double total_sessions, int64_t padding_idx, float* lse, float* z_pos,
                                         float* loss, void* ws, size_t ws_bytes, etpgt_stream_t stream_,
                                         int precision) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_precision("pool_softmax_fwd", precision);
  if (rc != ETPGT_OK) return rc;
  rc = pool_check_args(sess, table, targets, pool_ids, log_q, batch, num_items, num_sampled, dim, temperature,
                       padding_idx);
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(lse != nullptr && z_pos != nullptr && loss != nullptr,
                "pool_softmax_fwd: lse, z_pos and loss are required");
  Operands o;
  rc = pool_prepare(sess, table, targets, pool_ids, log_q, batch, num_sampled, dim, 1.f / temperature, padding_idx,
                    precision == ETPGT_SOFTMAX_BF16, z_pos, ws, ws_bytes, stream, &o);
  if (rc != ETPGT_OK) return rc;
  const double total = mean_over(total_sessions, batch);
  const Plan pl = plan_fwd(batch, num_sampled);
  Params p = call_params(dim, temperature, total, -1, o, nullptr);
  p.rows = batch;
  p.cols = num_sampled;
  p.tiles_per_range = pl.tiles_per_range;
  p.ranges = pl.ranges;
  rc = launch<FWD, true>(o.s_hi, o.s_lo, o.c_hi, o.c_lo, p, pl.grid, "pool_softmax_fwd", precision, stream);
  if (rc != ETPGT_OK) return rc;
  pool_combine_kernel<<<1, kCombineThreads, 0, stream>>>(o.part, pl.ranges, batch, z_pos, total, lse, loss);
  ETPGT_CHECK_LAUNCH("pool_softmax_fwd_combine");
  return ETPGT_OK;
}

extern "C" int etpgt_pool_softmax_fwd(const float* sess, const float* table, const int64_t* targets,
                                      const int64_t* pool_ids, const float* log_q, int64_t batch, int64_t num_items,
                                      int64_t num_sampled, int dim, float temperature, double total_sessions,
                                      int64_t padding_idx, float* lse, float* z_pos, float* loss, void* ws,
                                      size_t ws_bytes, etpgt_stream_t stream) {
  return etpgt_pool_softmax_fwd_ex(sess, table, targets, pool_ids, log_q, batch, num_items, num_sampled, dim,
                                   temperature, total_sessions, padding_idx, lse, z_pos, loss, ws, ws_bytes, stream,
                                   ETPGT_SOFTMAX_BF16X3);
}

extern "C" int etpgt_pool_softmax_bwd_ex(const float* sess, const float* table, const int64_t* targets,
                                         const int64_t* pool_ids, const float* log_q, const float* lse,
                                         const float* z_pos, const float* d_loss, int64_t batch, int64_t num_items,
                                         int64_t num_sampled, int dim, float temperature, double total_sessions,
                                         int64_t padding_idx, float* d_sess, float* d_table_accumulate, void* ws,
                                         size_t ws_bytes, etpgt_stream_t stream_, int precision) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  int rc = check_precision("pool_softmax_bwd", precision);
  if (rc != ETPGT_OK) return rc;
  rc = pool_check_args(sess, table, targets, pool_ids, log_q, batch, num_items, num_sampled, dim, temperature,
                       padding_idx);
  if (rc != ETPGT_OK) return rc;
  ETPGT_REQUIRE(lse != nullptr && z_pos != nullptr && d_loss != nullptr,
                "pool_softmax_bwd: lse, z_pos and d_loss are required");
  if (d_sess == nullptr && d_table_accumulate == nullptr) return ETPGT_OK;
  const bool bf16 = precision == ETPGT_SOFTMAX_BF16;
  Operands o;
  rc = pool_prepare(sess, table, targets, pool_ids, log_q, batch, num_sampled, dim, 1.f / temperature, padding_idx,
                    bf16, nullptr, ws, ws_bytes, stream, &o);
  if (rc != ETPGT_OK) return rc;
  const Params p = call_params(dim, temperature, mean_over(total_sessions, batch), -1, o, nullptr, lse, d_loss);
  if (d_sess != nullptr) {
    rc = grad_pass<DS, true>(o.s_hi, o.s_lo, o.c_hi, o.c_lo, p, batch, num_sampled, d_sess, 0, -1,
                             "pool_softmax_bwd_sess", "pool_softmax_bwd_sess_combine", precision, stream);
    if (rc != ETPGT_OK) return rc;
  }
  if (bf16)
    pool_positive_bwd_kernel<true><<<grid_for(batch, 8, 8), 256, 0, stream>>>(table, targets, z_pos, lse, d_loss,
                                                                              batch, dim, p.gscale, o.coef, d_sess);
  else
    pool_positive_bwd_kernel<<<grid_for(batch, 8, 8), 256, 0, stream>>>(table, targets, z_pos, lse, d_loss, batch,
                                                                        dim, p.gscale, o.coef, d_sess);
  ETPGT_CHECK_LAUNCH("pool_softmax_bwd_positive");
  if (d_table_accumulate != nullptr) {
    rc = grad_pass<DE, true>(o.c_hi, o.c_lo, o.s_hi, o.s_lo, p, num_sampled, batch, o.d_pool, 0, -1,
                             "pool_softmax_bwd_pool", "pool_softmax_bwd_pool_combine", precision, stream);
    if (rc != ETPGT_OK) return rc;
    // d_table[p_j] += d_pool[j], then d_table[t_b] += coef[b] s_b: each in ascending position, padding skipped
    rc = etpgt_scatter_rows(pool_ids, nullptr, o.d_pool, num_sampled, 1, dim, num_items, padding_idx,
                            d_table_accumulate, o.scatter_ws, o.scatter_bytes, stream);
    if (rc != ETPGT_OK) return rc;
    const float* s_rows = sess;
    if (bf16) {
      // bf16(s_b) as fp32 rows, in the session pair's slots (2 * s_pair >= batch * dim * 4 bytes): the passes that
      // read the bf16 sessions from there are done
      float* rounded = static_cast<float*>(o.s_slots);
      round_bf16_kernel<<<grid_for(batch * dim, 256, 8), 256, 0, stream>>>(sess, rounded, batch * dim);
      ETPGT_CHECK_LAUNCH("pool_softmax_bwd_round");
      s_rows = rounded;
    }
    rc = etpgt_scatter_rows(targets, o.coef, s_rows, batch, 1, dim, num_items, padding_idx, d_table_accumulate,
                            o.scatter_ws, o.scatter_bytes, stream);
    if (rc != ETPGT_OK) return rc;
  }
  return ETPGT_OK;
}

extern "C" int etpgt_pool_softmax_bwd(const float* sess, const float* table, const int64_t* targets,
                                      const int64_t* pool_ids, const float* log_q, const float* lse,
                                      const float* z_pos, const float* d_loss, int64_t batch, int64_t num_items,
                                      int64_t num_sampled, int dim, float temperature, double total_sessions,
                                      int64_t padding_idx, float* d_sess, float* d_table_accumulate, void* ws,
                                      size_t ws_bytes, etpgt_stream_t stream) {
  return etpgt_pool_softmax_bwd_ex(sess, table, targets, pool_ids, log_q, lse, z_pos, d_loss, batch, num_items,
                                   num_sampled, dim, temperature, total_sessions, padding_idx, d_sess,
                                   d_table_accumulate, ws, ws_bytes, stream, ETPGT_SOFTMAX_BF16X3);
}
