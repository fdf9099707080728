// a9: full-catalogue scoring on the 5th-generation tensor cores with a fused top-k epilogue.
//   scores[b, i] = <S[b, :], E[i, :]>  (bf16 operands, fp32 accumulation in TMEM), top-k per row
// etpgt/model/base.py:59-78 (`torch.matmul(S, E.t())` + `torch.topk`).  The [B, I] score matrix is
// never written.
//
// GEMM kernel (one CTA = 128 sessions x a contiguous range of 256-item tiles; CTA pairs: 256 sessions):
//   warp 0      TMA producer: session tile once (DIM/64 k-blocks of 128x64 bf16, SWIZZLE_128B), then
//               a ring of item k-blocks (256x64 bf16; a pair: 128x64 per CTA) with mbarrier full/empty hand-shakes
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer (UMMA 128x256x16, a pair: 256x256x16 issued by
//               the leader; kind::f16), accumulators double-buffered in the 512 TMEM columns
//   warps 2-9   epilogue: two warps per TMEM lane quarter (lane = session row), one per column half of a tile
//
// Epilogue = "piece dump".  Measured on B200: with an epilogue that only loads TMEM and takes
// maxima the pipeline runs at 84 % of the cuBLAS bf16 peak; every form of per-item candidate
// handling inside the loop (shared-memory k-lists: 3 %, pending buffers: 23 %, register lists with
// warp-uniform scans: 30 %) was bound by SIMT divergence — the 32 rows of a warp accept candidates
// at different columns, so each accepted item costs the whole warp an insert.  So the loop keeps,
// per row, only the K best 16-column PIECE MAXIMA in a register-resident sorting network (values
// only, branch-free, all lanes in lockstep), and a lane whose piece maximum beats its row's
// threshold dumps that piece's 16 raw scores (64 bytes) to a per-(row, range) slot buffer in HBM.
// K piece maxima >= thr prove K items >= thr, so thr is a valid lower bound of the row's K-th best
// score and no piece holding a top-K item is ever skipped (a warp sees its pieces in ascending id
// order and the test is a strict '>', so ties keep the lower id).
//
// At K = 256 an accumulator element receives only 16 MMAs: a 128 x 256 tile is produced in ~2,000
// cycles, while ONE warp per TMEM lane quarter needed ~4,100 (round 1: ~790 instructions per tile
// at ~5 cycles each — a single warp per scheduler cannot hide its own latencies).  So TWO warps
// work on every lane quarter, columns 0-127 / 128-255 of each tile, each with its own sorted list,
// threshold and pending buffer; they fill the row's slot buffer from both ends (no shared counter)
// and read each other's threshold through shared memory (a piece must also reach the OTHER warp's
// threshold — '>=' there, because that warp's pieces may have higher ids).  About 200-250 pieces
// (14 KB) per row are dumped.  (A variant with the lists kept by separate merge warps in shared
// memory was measured and dropped: whenever the merge fell behind, the thresholds went stale, more
// pieces qualified and the merge fell further behind — 630-1,700 pieces per row.)
//
// CTA pairs (default): two CTAs on the two SMs of a TPC execute ONE tcgen05.mma of M = 256 (cta_group::2).  Each
// keeps its own 128 session rows resident and loads only HALF of every item k-block (128 of the 256 item rows);
// the tensor cores of both SMs read both halves, so the L2 -> shared-memory traffic per SM — 62 B/clk at the full
// MMA rate against ~43 B/clk per SM that the L2 sustains chip-wide — halves, and a stage shrinks to 16 KB (six
// stages).  The leader (cluster rank 0) issues the MMAs and commits to the barriers of both CTAs (multicast); each
// CTA's eight epilogue warps drain their own 128 accumulator rows and release the accumulator stage on the leader's
// barrier (16 arrivals).  An epilogue warp loads three of its four 32-column chunks to registers at once, the
// fourth into the first one's registers once that is worked off, and hands the accumulator back BEFORE it works
// on the rest and before the lockstep merge: the MMA issuer never waits for a warp that is busy merging.
// Measured (23,861 x 82,174 x 256, top-20): 0.96 ms (round 1: one CTA per unit, one epilogue warp per quarter)
// -> 0.85-0.87 ms; GEMM kernel alone 0.75 ms with the tensor pipe 72 % active (ncu), select 0.08 ms.
//
// Select kernel (one warp per row): reads the 8-byte records (first column, maximum) of the row's dumped pieces,
// keeps the pieces whose maximum reaches the best threshold of the row's ranges / column halves (a few dozen of
// ~215), reads only those (two pieces per warp step, one score per lane) and picks the exact top-k by (score desc,
// id asc) with a bitonic sort of 64-bit keys in registers.  Rows whose slot buffer overflowed (adversarial score
// orders) are recomputed exactly by a CUDA-core fallback kernel, so the result is always exact.
//
// Exclusion (etpgt_score_topk_bf16_exclude, the EXCL variant): every row may name item ids it must not receive (the
// session's own items, the padding id).  The epilogue sets those columns to -inf BEFORE the piece maxima are taken:
// an excluded item holding one of the K best piece maxima would otherwise raise the threshold above the K-th best
// ELIGIBLE score, and the pieces that hold the eligible top-k would never be dumped.  Each epilogue thread walks its
// row's ascending list with one cursor; per 32-column chunk that costs one compare, and only the few chunks that
// contain an excluded id (about 6 per row at 82k items) take the masking branch.  Dumped pieces carry the -inf, the
// select kernel never keeps a -inf score and the fallback kernel skips the listed ids, so a row with fewer than k
// eligible items ends in (-inf, INT64_MAX) sentinels.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "tc_common.cuh"

namespace etpgt {
namespace {

using namespace tc;

constexpr int BLOCK_M = 128;   // sessions per CTA (TMEM lanes)
constexpr int BLOCK_N = 256;   // items per accumulator tile (TMEM columns)
constexpr int CHUNK = 32;      // columns per tcgen05.ld
constexpr int DUMPW = 16;      // columns per dumped piece (64 bytes)
constexpr int kMaxStages = 6;  // ring of item k-blocks (3 of 32 KB per CTA, 6 of 16 KB per CTA of a pair)
constexpr int kAccStages = 2;  // TMEM accumulator double buffer
constexpr int kTmemCols = 512;
constexpr int kMaxColParts = 4;     // epilogue warps per TMEM lane quarter (each takes 256 / parts columns of a tile)
constexpr int threads_for(int col_parts) { return 32 * (2 + 4 * col_parts); }
constexpr int kMaxKTc = 32;
constexpr int kPendingMerge = 16;  // capacity: maxima a row may have waiting (merge threshold - 1 + pieces per tile half)
constexpr int kDefaultPendingMerge = 8;
constexpr uint32_t A_KBLOCK_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB
constexpr uint32_t B_STAGE_BYTES = BLOCK_N * BLOCK_K * 2;   // 32 KB (a pair: 16 KB in each CTA)

struct __align__(8) Barriers {
  uint64_t a_full;
  uint64_t b_full[kMaxStages];
  uint64_t b_empty[kMaxStages];
  uint64_t acc_full[kAccStages];
  uint64_t acc_empty[kAccStages];
  uint32_t tmem_base;
};

// Shared-memory scratch of the epilogue warps.
struct RowShared {
  float pending[4 * kMaxColParts][kPendingMerge][32];  // piece maxima waiting for the warp's lockstep merge
  float thr[kMaxColParts][BLOCK_M];                    // [column part][row]: that warp's current threshold
};

// Dump buffers, per (row, range): `cap` slots of 32 scores + the chunk's first column (relative to the
// range), a slot count (may exceed cap = overflow) and the range's final threshold.
struct DumpBuffers {
  float* scores;      // [rows*splits][cap][DUMPW]
  int2* meta;         // [rows*splits][cap]: (first column of the piece relative to the range, bits of the piece's
                      // maximum) — the select kernel reads these first
  int32_t* count;     // [col_parts][rows*splits]: pieces dumped by each column part
  float* threshold;   // [col_parts][rows*splits]: final threshold of each column part
  int64_t units;      // rows*splits
  int cap;            // slots per (row, range) = (col_parts / 2) sub-buffers of cap_sub slots; two column parts share a
  int cap_sub;        // sub-buffer and fill it from both ends (no shared counter)
  int col_parts;
};

// Work units.  One CTA per SM and one long range per row is the cheapest (every range pays a warm-up
// while its thresholds rise from -inf), but the number of 128-row tiles is rarely a multiple of 148.
// So the first `m_full` row tiles (whole waves) each scan the WHOLE catalogue as one unit, and only
// the remaining row tiles are cut into `tail_splits` item ranges to fill the last wave.
struct Schedule {
  int m_full;           // row tiles with a single full-catalogue unit (a multiple of the worker count, may be 0)
  int tail_splits;      // item ranges per remaining row tile
  int tiles_per_split;  // 256-item tiles per tail range
  int total_tiles;
  int unit_rows;        // rows of a row tile: 128 (one CTA) or 256 (a CTA pair)
  __host__ __device__ int64_t full_rows() const { return (int64_t)m_full * unit_rows; }
  __host__ __device__ int parts_of_row(int64_t row) const { return row < full_rows() ? 1 : tail_splits; }
  // index of (row, part) in the count / threshold arrays; x cap in the slot arrays
  __host__ __device__ int64_t part_index(int64_t row, int part) const {
    return row < full_rows() ? row : full_rows() + (row - full_rows()) * tail_splits + part;
  }
  __host__ __device__ int first_tile(int64_t row, int part) const { return row < full_rows() ? 0 : part * tiles_per_split; }
  __host__ __device__ int64_t num_parts(int64_t batch) const {
    const int64_t f = batch < full_rows() ? batch : full_rows();
    return f + (batch - f) * tail_splits;
  }
};

// Exclusion lists: ids [batch, width], each row ascending (duplicates allowed); ids outside [id_base, id_base +
// num_items) are ignored, so an item shard takes the global list unchanged and -1 pads a row.
struct Exclusion {
  const int64_t* ids;
  int64_t width;
  int64_t id_base;
};
constexpr int64_t kMaxExcludeWidth = 16384;   // the fallback kernel stages a row's list in shared memory

// One epilogue thread's cursor into its row's list.  Only the next entry's column (relative to the thread's range;
// INT_MAX once the list is used up) stays in a register: the hot loop compares against it once per chunk.  The rest
// is read on the rare masking path only, so it lives in shared memory (in registers it made ptxas spill).
struct ExclCursor {
  const int64_t* next;
  int64_t base;   // id of the range's column 0
  int left;       // entries from `next` on
};

__device__ __forceinline__ int excl_col(int64_t id, int64_t base) {
  const int64_t c = id - base;   // >= 0: ids below the range were skipped by a lower bound
  return c < (int64_t)INT_MAX ? (int)c : INT_MAX;
}

// Per-row state of the piece-dump epilogue (one thread = one session row = one TMEM lane, one column half).
template <int KCAP>
struct RowState {
  float best[KCAP];   // the KCAP largest piece maxima of this row (this half) so far, descending
  float thr;          // = best[KCAP - 1] as of the last merge: a lower bound of the row's K-th best score
  int count, pending;
};

// One 32-column chunk of a row: piece maxima, dump of the pieces that beat the thresholds; their maxima wait in the
// warp's pending buffer for the merge at the end of the tile.
//   slot_first / slot_step: this warp fills the slot buffer upwards from 0 or downwards from cap - 1
// (The hot loop has to stay inside the instruction cache: with four inlined copies of chunk + merge ncu showed 1.8
// "no instruction" stall cycles per issued instruction; the merge exists once per kernel now.)
template <int KCAP, bool EXCL>
__device__ __forceinline__ void chunk_hits(const uint32_t (&raw)[CHUNK], RowState<KCAP>& st, int col,
                                           int limit_rel /* real columns left from this chunk on */,
                                           float* my_scores, int2* my_meta, int cap, int slot_first, int slot_step,
                                           uint32_t my_pending,
                                           float thr_other /* a little stale at worst: still a valid bound */,
                                           int& ex_col, ExclCursor* ex) {
  float v[CHUNK];
#pragma unroll
  for (int j = 0; j < CHUNK; ++j) v[j] = __uint_as_float(raw[j]);
  if (limit_rel < CHUNK) {  // only the table's last tile: columns past the end never qualify
#pragma unroll
    for (int j = 0; j < CHUNK; ++j) v[j] = j < limit_rel ? v[j] : -INFINITY;
  }
  if (EXCL && ex_col < col + CHUNK) {   // rare: the row's next excluded id lies in (or before) this chunk
    const int64_t* next = ex->next;
    const int64_t base = ex->base;
    int left = ex->left;
    do {
      const int e = ex_col - col;         // < 0: an id among another column part's columns, nothing to mask here
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) v[j] = j == e ? -INFINITY : v[j];   // a select, no dynamic register index
      ++next;
      --left;
      ex_col = left > 0 ? excl_col(*next, base) : INT_MAX;
    } while (ex_col < col + CHUNK);
    ex->next = next;
    ex->left = left;
  }
  float g[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) g[q] = fmaxf(fmaxf(v[4 * q], v[4 * q + 1]), fmaxf(v[4 * q + 2], v[4 * q + 3]));
  // dump granularity = DUMPW (16) columns: one 64-byte piece per hit instead of the whole 128-byte
  // chunk — a third less dump traffic and half the store instructions on the divergent path
  float mx[CHUNK / DUMPW];
  bool hit[CHUNK / DUMPW];
  bool any_hit = false;
#pragma unroll
  for (int h = 0; h < CHUNK / DUMPW; ++h) {
    mx[h] = fmaxf(fmaxf(g[4 * h], g[4 * h + 1]), fmaxf(g[4 * h + 2], g[4 * h + 3]));
    hit[h] = mx[h] > st.thr && mx[h] >= thr_other;   // rows past the batch carry thr = +inf
    any_hit = any_hit || hit[h];
  }
  if (!__any_sync(0xffffffffu, any_hit)) return;  // warp-uniform
#pragma unroll
  for (int h = 0; h < CHUNK / DUMPW; ++h) {
    if (hit[h]) {
      const int n = st.count++;
      st_shared_f32(my_pending + st.pending * 32 * sizeof(float), mx[h]);  // waits for the lockstep merge
      ++st.pending;
      if (n < cap) {
        const int slot = slot_first + slot_step * n;
        my_meta[slot] = make_int2(col + h * DUMPW, __float_as_int(mx[h]));
        float4* dst = reinterpret_cast<float4*>(my_scores + (int64_t)slot * DUMPW);
#pragma unroll
        for (int q = 0; q < DUMPW / 4; ++q) {
          const int j = h * DUMPW + 4 * q;
          __stcs(dst + q, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
        }
      }
    }
  }
}

// Merge the pending piece maxima of all 32 rows into the sorted lists TOGETHER: one pass of the sorting network
// then serves up to 32 rows at once (run per hit it would serve ~1).  The threshold is a little stale in between,
// which only dumps a few extra pieces.
template <int KCAP>
__device__ __forceinline__ void merge_pending(RowState<KCAP>& st, uint32_t my_pending, uint32_t thr_own_addr,
                                              int pending_merge) {
  if (!__any_sync(0xffffffffu, st.pending >= pending_merge)) return;
  int most = st.pending;
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) most = max(most, __shfl_xor_sync(0xffffffffu, most, off));
#pragma unroll 2
  for (int p = 0; p < most; ++p) {
    float x = p < st.pending ? ld_shared_f32(my_pending + p * 32 * sizeof(float)) : -INFINITY;  // -inf: no-op
#pragma unroll
    for (int s = 0; s < KCAP; ++s) {
      const float hi = fmaxf(st.best[s], x);
      x = fminf(st.best[s], x);
      st.best[s] = hi;
    }
  }
  st.pending = 0;
  st.thr = st.best[KCAP - 1];
  st_shared_f32(thr_own_addr, st.thr);
}

// NUM_KB = DIM / 64; KCAP = piece maxima tracked per row and column part (>= k); PAIR = CTA pairs; CP = column parts;
// EXCL = the rows' exclusion lists are applied (`excl` is ignored otherwise)
template <int NUM_KB, int KCAP, bool PAIR, int CP, bool EXCL>
__global__ void __launch_bounds__(threads_for(CP), 1)
score_dump_tc_kernel(const __grid_constant__ CUtensorMap map_sess, const __grid_constant__ CUtensorMap map_items,
                     int64_t batch, int64_t num_items, int stages, Schedule sch, DumpBuffers dump,
                     int pending_merge /* <= kPendingMerge */, Exclusion excl) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  constexpr int LOAD_N = PAIR ? BLOCK_N / 2 : BLOCK_N;          // item rows this CTA loads per k-block
  constexpr uint32_t STAGE_BYTES = LOAD_N * BLOCK_K * 2;
  constexpr uint32_t kInstrDesc = instr_desc_bf16(PAIR ? 2 * BLOCK_M : BLOCK_M, BLOCK_N);
  uint8_t* smem_a = smem;                                   // NUM_KB x 16 KB
  uint8_t* smem_b = smem_a + NUM_KB * A_KBLOCK_BYTES;       // stages x STAGE_BYTES
  RowShared* rs = reinterpret_cast<RowShared*>(smem_b + stages * STAGE_BYTES);
  Barriers* bars = reinterpret_cast<Barriers*>(rs + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0;       // 0 = the pair's leader
  const int unit = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  int m_unit, part;
  int64_t tile_begin, tile_end;
  if (unit < sch.m_full) {
    m_unit = unit; part = 0; tile_begin = 0; tile_end = sch.total_tiles;
  } else {
    const int v = unit - sch.m_full;
    m_unit = sch.m_full + v / sch.tail_splits;
    part = v % sch.tail_splits;
    tile_begin = (int64_t)part * sch.tiles_per_split;
    tile_end = tile_begin + sch.tiles_per_split < sch.total_tiles ? tile_begin + sch.tiles_per_split : sch.total_tiles;
  }
  const int m_tile = PAIR ? 2 * m_unit + (int)rank : m_unit;   // this CTA's 128 session rows
  const int num_tiles = tile_end > tile_begin ? (int)(tile_end - tile_begin) : 0;

  if (threadIdx.x == 0) {
    // barriers that gate the MMAs count the producers of BOTH CTAs and live in the leader
    mbar_init(&bars->a_full, PAIR ? 2 : 1);
    for (int s = 0; s < kMaxStages; ++s) { mbar_init(&bars->b_full[s], PAIR ? 2 : 1); mbar_init(&bars->b_empty[s], 1); }
    for (int s = 0; s < kAccStages; ++s) {
      mbar_init(&bars->acc_full[s], 1);
      mbar_init(&bars->acc_empty[s], PAIR ? 2 * 4 * CP : 4 * CP);
    }
    fence_barrier_init();
    tma_prefetch_desc(&map_sess);
    tma_prefetch_desc(&map_items);
  }
  for (int i = threadIdx.x; i < kMaxColParts * BLOCK_M; i += threads_for(CP)) (&rs->thr[0][0])[i] = -INFINITY;
  if (warp == 1) {
    if (PAIR) tmem_alloc_2sm(&bars->tmem_base, kTmemCols);
    else tmem_alloc(&bars->tmem_base, kTmemCols);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // both CTAs' barriers are initialised before anything crosses the pair
  tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ===================== TMA producer (one elected lane; in a pair: of each CTA) =====================
    if (lane == 0 && num_tiles > 0) {
      if (PAIR) {
        const uint32_t a_full = mapa_shared(smem_u32(&bars->a_full), 0);
        mbar_arrive_expect_tx_cluster(a_full, NUM_KB * A_KBLOCK_BYTES);
        for (int kb = 0; kb < NUM_KB; ++kb)
          tma_load_2d_2sm(&map_sess, a_full, smem_a + kb * A_KBLOCK_BYTES, kb * BLOCK_K, m_tile * BLOCK_M);
      } else {
        mbar_expect_tx(&bars->a_full, NUM_KB * A_KBLOCK_BYTES);
        for (int kb = 0; kb < NUM_KB; ++kb)
          tma_load_2d(&map_sess, &bars->a_full, smem_a + kb * A_KBLOCK_BYTES, kb * BLOCK_K, m_tile * BLOCK_M);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < num_tiles; ++t) {
        const int row0 = (int)((tile_begin + t) * BLOCK_N) + (int)rank * LOAD_N;   // a pair: this CTA's half
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait(&bars->b_empty[stage], phase ^ 1);
          if (PAIR) {
            const uint32_t full = mapa_shared(smem_u32(&bars->b_full[stage]), 0);
            mbar_arrive_expect_tx_cluster(full, STAGE_BYTES);
            tma_load_2d_2sm(&map_items, full, smem_b + stage * STAGE_BYTES, kb * BLOCK_K, row0);
          } else {
            mbar_expect_tx(&bars->b_full[stage], STAGE_BYTES);
            tma_load_2d(&map_items, &bars->b_full[stage], smem_b + stage * STAGE_BYTES, kb * BLOCK_K, row0);
          }
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (one elected lane; in a pair: of the leader) =====================
    if (lane == 0 && rank == 0 && num_tiles > 0) {
      mbar_wait(&bars->a_full, 0);
      tc_fence_after();
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < num_tiles; ++t) {
        const int acc = t & 1;
        const uint32_t acc_phase = (uint32_t)(t >> 1) & 1;
        mbar_wait(&bars->acc_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = 0; kb < NUM_KB; ++kb) {
          mbar_wait(&bars->b_full[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + kb * A_KBLOCK_BYTES);
          const uint32_t b_addr = smem_u32(smem_b + stage * STAGE_BYTES);
#pragma unroll
          for (int kk = 0; kk < BLOCK_K / UMMA_K; ++kk) {
            const uint64_t da = make_desc_sw128(a_addr + kk * UMMA_K * 2);
            const uint64_t db = make_desc_sw128(b_addr + kk * UMMA_K * 2);
            if (PAIR) umma_bf16_2sm(tmem_d, da, db, kInstrDesc, (kb | kk) != 0 ? 1u : 0u);
            else umma_bf16(tmem_d, da, db, kInstrDesc, (kb | kk) != 0 ? 1u : 0u);
          }
          // frees the smem stage (in both CTAs) once these MMAs have read it
          if (PAIR) umma_commit_2sm(&bars->b_empty[stage]);
          else umma_commit(&bars->b_empty[stage]);
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        // accumulator tile complete (each CTA's epilogue reads its own 128 rows from its own TMEM)
        if (PAIR) umma_commit_2sm(&bars->acc_full[acc]);
        else umma_commit(&bars->acc_full[acc]);
      }
    }
  } else {
    // ========== epilogue: 4 * CP warps; TMEM lane quarter = warp % 4, column part = (warp - 2) / 4 ==========
    const int quarter = warp & 3;
    const int cpart = (warp - 2) >> 2;
    const int row = quarter * 32 + lane;       // session row inside the tile == TMEM lane
    const int64_t grow = (int64_t)m_tile * BLOCK_M + row;
    const bool live = grow < batch;
    const int64_t pidx = live ? sch.part_index(grow, part) : 0;
    const int64_t slot0 = pidx * (int64_t)dump.cap + (cpart >> 1) * dump.cap_sub;   // this pair of parts' sub-buffer
    float* my_scores = dump.scores + slot0 * DUMPW;
    int2* my_meta = dump.meta + slot0;
    RowState<KCAP> st;
#pragma unroll
    for (int t = 0; t < KCAP; ++t) st.best[t] = live ? -INFINITY : INFINITY;   // rows past the batch never qualify
    st.thr = st.best[KCAP - 1];
    st.count = 0;
    st.pending = 0;
    const uint32_t my_pending = smem_u32(&rs->pending[warp - 2][0][lane]);
    const uint32_t thr_row_addr = smem_u32(&rs->thr[0][row]);
    const uint32_t thr_own_addr = thr_row_addr + (uint32_t)(cpart * BLOCK_M * sizeof(float));
    const uint32_t acc_empty0 = PAIR ? mapa_shared(smem_u32(&bars->acc_empty[0]), 0) : smem_u32(&bars->acc_empty[0]);
    constexpr int PART_N = BLOCK_N / CP;
    // loop constants pinned in registers (as kernel parameters they were re-read from the constant bank on the
    // divergent path: ~2 % of the epilogue's stall samples)
    int cap = dump.cap_sub, merge_at = pending_merge;
    int slot_first = (cpart & 1) ? dump.cap_sub - 1 : 0, slot_step = (cpart & 1) ? -1 : 1;
    asm volatile("" : "+r"(cap), "+r"(merge_at), "+r"(slot_first), "+r"(slot_step));
    // exclusion cursor: starts at the lower bound of the range's first id in the row's list
    ExclCursor* ex = reinterpret_cast<ExclCursor*>(bars + 1) + (threadIdx.x - 64);
    int ex_col = INT_MAX;
    if (EXCL && live) {
      const int64_t base = excl.id_base + tile_begin * BLOCK_N;
      const int64_t* ids = excl.ids + grow * excl.width;
      int lo = 0, hi = (int)excl.width;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (ids[mid] < base) lo = mid + 1;
        else hi = mid;
      }
      *ex = ExclCursor{ids + lo, base, (int)excl.width - lo};
      ex_col = lo < excl.width ? excl_col(ids[lo], base) : INT_MAX;
    }
    for (int t = 0; t < num_tiles; ++t) {
      const int acc = t & 1;
      const uint32_t acc_phase = (uint32_t)(t >> 1) & 1;
      mbar_wait(&bars->acc_full[acc], acc_phase);
      tc_fence_after();
      const int64_t item0 = (tile_begin + t) * BLOCK_N + cpart * PART_N;
      const int limit = num_items - item0 < PART_N ? (int)(num_items - item0) : PART_N;  // real columns of this part
      const int col0 = t * BLOCK_N + cpart * PART_N;
      const uint32_t taddr =
          tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BLOCK_N + cpart * PART_N);
      // This warp's columns of the tile go to registers as early as the register file allows (all chunks but one,
      // the last into the first one's registers once that is worked off) and the accumulator
      // is handed back before the rest is processed and before any merge: the MMA issuer (which needs every epilogue
      // warp — of both CTAs of a pair — to let go) no longer waits for a warp that is busy in a lockstep merge.
      constexpr int NCH = PART_N / CHUNK;             // 4 or 2
      constexpr int NBUF = NCH - 1;                   // 3 or 1 (96 registers per thread with 18 warps)
      uint32_t raw[NBUF][CHUNK];
#pragma unroll
      for (int c = 0; c < NBUF; ++c) tmem_ld_32x32_issue(taddr + (uint32_t)(c * CHUNK), raw[c]);
      // the other column parts' thresholds: a little stale at worst, still valid bounds
      float thr_other = -INFINITY;
#pragma unroll
      for (int o = 1; o < CP; ++o)
        thr_other = fmaxf(thr_other, ld_shared_f32(thr_row_addr + (uint32_t)(((cpart + o) % CP) * BLOCK_M * sizeof(float))));
#pragma unroll
      for (int c = 0; c < NBUF; ++c) tmem_ld_wait(raw[c]);
      if (NCH > NBUF) {
        chunk_hits<KCAP, EXCL>(raw[0], st, col0, limit, my_scores, my_meta, cap, slot_first, slot_step, my_pending,
                               thr_other, ex_col, ex);
        tmem_ld_32x32(taddr + (uint32_t)(NBUF * CHUNK), raw[0]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster(acc_empty0 + (uint32_t)(acc * sizeof(uint64_t)));
        else mbar_arrive(&bars->acc_empty[acc]);
      }
      // the lockstep merge (long: up to 15 passes of the sorting network) comes AFTER the hand-back, so that it never
      // sits between an accumulator becoming ready and this warp letting go of it
      merge_pending<KCAP>(st, my_pending, thr_own_addr, merge_at);
#pragma unroll
      for (int c = NCH > NBUF ? 1 : 0; c < NCH; ++c)
        chunk_hits<KCAP, EXCL>(raw[c % NBUF], st, col0 + c * CHUNK, limit - c * CHUNK, my_scores, my_meta, cap,
                               slot_first, slot_step, my_pending, thr_other, ex_col, ex);
    }
    merge_pending<KCAP>(st, my_pending, thr_own_addr, 1);   // what is still waiting: the final threshold
    if (live) {
      dump.count[(int64_t)cpart * dump.units + pidx] = st.count;
      dump.threshold[(int64_t)cpart * dump.units + pidx] = st.thr;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // neither CTA's shared memory / TMEM goes away while the other still uses it
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2sm(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
}

__device__ __forceinline__ bool better(float v, int64_t i, float bv, int64_t bi) {
  return v > bv || (v == bv && i < bi);
}

// (score, column) packed so that an unsigned 64-bit comparison orders candidates by score descending,
// then column ascending: high word = order-preserving image of the float (-0.0 canonicalised to +0.0,
// like the oracle's comparison), low word = ~column.  0 is never a valid key.
__device__ __forceinline__ uint64_t candidate_key(float v, int32_t col) {
  uint32_t f = __float_as_uint(v + 0.0f);
  f = (f & 0x80000000u) ? ~f : (f | 0x80000000u);
  return ((uint64_t)f << 32) | (uint64_t)(0xFFFFFFFFu - (uint32_t)col);
}
__device__ __forceinline__ void decode_key(uint64_t key, float& v, int64_t& col) {
  if (key == 0) { v = -INFINITY; col = 0; return; }
  const uint32_t f = (uint32_t)(key >> 32);
  v = __uint_as_float((f & 0x80000000u) ? (f ^ 0x80000000u) : ~f);
  col = (int64_t)(0xFFFFFFFFu - (uint32_t)key);
}

// One warp per row.  Survivors (scores >= the best range threshold) are collected in shared memory as
// packed keys, then sorted (bitonic network over 64 keys; selection passes when there are more).
constexpr int kSelectWarps = 4;
constexpr int kSurvivorCap = 512;
constexpr int kFlagCap = 256;        // qualifying pieces per row (more: the row goes to the exact fallback)

__global__ void __launch_bounds__(kSelectWarps * 32)
score_select_kernel(DumpBuffers dump, int64_t batch, Schedule sch, int k, int64_t id_base,
                    float* __restrict__ top_val, int64_t* __restrict__ top_idx, int32_t* __restrict__ redo,
                    const int64_t* __restrict__ targets, int32_t* __restrict__ hit_pos) {
  __shared__ uint64_t s_key[kSelectWarps][kSurvivorCap];  // (orderable score, ~column): larger = better
  __shared__ int2 s_flag[kSelectWarps][kFlagCap];          // qualifying pieces: (slot relative to the row's first, column)
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * (int64_t)kSelectWarps + w;
  if (row >= batch) return;
  int n_flag = 0, n_surv = 0;                               // warp-uniform counters
  const int64_t row_slot0 = sch.part_index(row, 0) * (int64_t)dump.cap;
  float tau = -INFINITY;
  bool overflow = false;
  const int splits = sch.parts_of_row(row);
  const int cparts = dump.col_parts;
  for (int s = 0; s < splits; ++s) {
    const int64_t pi = sch.part_index(row, s);
    for (int c = 0; c < cparts; c += 2) {
      tau = fmaxf(tau, fmaxf(dump.threshold[c * dump.units + pi], dump.threshold[(c + 1) * dump.units + pi]));
      overflow = overflow || dump.count[c * dump.units + pi] + dump.count[(c + 1) * dump.units + pi] > dump.cap_sub;
    }
  }
  __syncwarp();
  if (!overflow) {
    for (int seg = 0; seg < cparts * splits; ++seg) {
      // a (row, range) slot buffer is col_parts / 2 sub-buffers, each filled from both ends by two column parts
      const int s = seg / cparts, c = seg % cparts;
      const int64_t pi = sch.part_index(row, s);
      const int n = dump.count[c * dump.units + pi];
      const int64_t slot0 = pi * (int64_t)dump.cap + (c >> 1) * dump.cap_sub + ((c & 1) ? dump.cap_sub - n : 0);
      const int range_col0 = sch.first_tile(row, s) * BLOCK_N;
      // the piece maxima first (one coalesced 8-byte load per piece): the pieces that reach tau — a few dozen of the
      // ~200 dumped per row — are collected as (slot, first column) pairs ...
      const int2* meta = dump.meta + slot0;
      for (int c0 = 0; c0 < n; c0 += 128) {
        int2 m[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          m[u] = c0 + 32 * u + lane < n ? __ldcs(meta + c0 + 32 * u + lane) : make_int2(0, (int)0xff800000u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float pm = __int_as_float(m[u].y);
          const bool flag = pm >= tau && pm > -INFINITY;
          const unsigned mask = __ballot_sync(0xffffffffu, flag);
          if (flag) {
            const int pos = n_flag + __popc(mask & ((1u << lane) - 1));
            if (pos < kFlagCap) s_flag[w][pos] = make_int2((int)(slot0 - row_slot0) + c0 + 32 * u + lane, range_col0 + m[u].x);
          }
          n_flag += __popc(mask);
        }
      }
    }
    __syncwarp();
    if (n_flag > kFlagCap) {
      overflow = true;
    } else {
      // ... and read two at a time: half a warp per piece, one score per lane (a coalesced 64-byte line)
      const int sub = lane >> 4, e = lane & 15;
      for (int f0 = 0; f0 < n_flag; f0 += 8) {      // four independent loads in flight per lane
        int2 fl[4];
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool have = f0 + 2 * u + sub < n_flag;
          fl[u] = have ? s_flag[w][f0 + 2 * u + sub] : make_int2(0, 0);
          v[u] = have ? __ldcs(dump.scores + (row_slot0 + fl[u].x) * DUMPW + e) : -INFINITY;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const bool keep = v[u] >= tau && v[u] > -INFINITY;   // -inf: past the table's end, or an excluded id
          const unsigned mask = __ballot_sync(0xffffffffu, keep);
          if (keep) {
            const int pos = n_surv + __popc(mask & ((1u << lane) - 1));
            if (pos < kSurvivorCap) s_key[w][pos] = candidate_key(v[u], fl[u].y + e);
          }
          n_surv += __popc(mask);
        }
      }
      __syncwarp();
      overflow = n_surv > kSurvivorCap;  // a huge tie at the threshold
    }
  }
  if (overflow) {
    if (lane == 0) redo[row] = 1;
    return;
  }
  if (lane == 0) redo[row] = 0;
  const int n = n_surv;
  uint64_t mine = 0;   // lane t ends up with the t-th best candidate (0 = none)
  if (n <= 32) {
    // a bitonic sort of 32 keys, one per lane, descending
    uint64_t k0 = lane < n ? s_key[w][lane] : 0;
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const uint64_t p0 = __shfl_xor_sync(0xffffffffu, k0, stride);
        const bool lower = (lane & stride) == 0;
        const bool desc = size == 32 || ((lane & size) == 0);
        k0 = (lower == desc) ? (k0 > p0 ? k0 : p0) : (k0 < p0 ? k0 : p0);
      }
    }
    mine = k0;
  } else if (n <= 64) {
    // a few dozen survivors: bitonic sort of 64 keys, two per lane, descending
    uint64_t k0 = lane < n ? s_key[w][lane] : 0, k1 = lane + 32 < n ? s_key[w][lane + 32] : 0;
#pragma unroll
    for (int size = 2; size <= 64; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        if (stride == 32) {          // partner of element i (< 32) is i + 32: the lane's own second key
          const uint64_t hi = k0 > k1 ? k0 : k1, lo = k0 > k1 ? k1 : k0;   // size == 64: descending everywhere
          k0 = hi; k1 = lo;
        } else {
          // element index e0 = lane, e1 = lane + 32; direction of the bitonic block containing the element
          const uint64_t p0 = __shfl_xor_sync(0xffffffffu, k0, stride), p1 = __shfl_xor_sync(0xffffffffu, k1, stride);
          const bool lower = (lane & stride) == 0;                       // this lane holds the lower index of the pair
          const bool desc0 = size == 64 || ((lane & size) == 0);        // block direction (final merge: descending)
          const bool desc1 = size == 64 || (((lane + 32) & size) == 0);
          const bool take_max0 = lower == desc0, take_max1 = lower == desc1;
          k0 = take_max0 ? (k0 > p0 ? k0 : p0) : (k0 < p0 ? k0 : p0);
          k1 = take_max1 ? (k1 > p1 ? k1 : p1) : (k1 < p1 ? k1 : p1);
        }
      }
    }
    mine = k0;                       // ranks 0..31 are the first keys of lanes 0..31 (k <= 32)
  } else {
    // many survivors (large ties at the threshold): k selection passes over the shared-memory list
    uint64_t prev = ~uint64_t(0);
    for (int t = 0; t < k; ++t) {
      uint64_t best = 0;
      for (int c = lane; c < n; c += 32) {
        const uint64_t key = s_key[w][c];
        if (key < prev && key > best) best = key;
      }
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        const uint64_t o = __shfl_xor_sync(0xffffffffu, best, off);
        best = o > best ? o : best;
      }
      if (lane == t) mine = best;
      prev = best;
    }
  }
  float v;
  int64_t col;
  decode_key(mine, v, col);
  const int64_t id = mine == 0 ? INT64_MAX : id_base + col;
  if (lane < k) {   // one coalesced store of the row's k results
    top_val[row * k + lane] = v;
    top_idx[row * k + lane] = id;
  }
  if (targets != nullptr) {
    // Recall / NDCG input (etpgt/utils/metrics.py:6-66) straight from the registers that hold the sorted list:
    // position of the row's target among its k results (first match), or -1
    const unsigned found = __ballot_sync(0xffffffffu, lane < k && id == targets[row]);
    if (lane == 0) hit_pos[row] = found ? __ffs(found) - 1 : -1;
  }
}

// Exact CUDA-core recomputation of the rows flagged in `redo` (slot-buffer or tie overflow): one CTA
// per row, every thread scores a strided share of the items (fp32 accumulation of the same bf16
// operands) and keeps a private sorted k-list; lists are merged through shared memory.
// EXCL: the row's exclusion list is staged in shared memory and an item that would enter a list is
// looked up there first (a binary search; rare once the lists have filled).
constexpr int kRedoThreads = 256;

__device__ __forceinline__ bool listed(const int64_t* ids, int n, int64_t id) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (ids[mid] < id) lo = mid + 1;
    else hi = mid;
  }
  return lo < n && ids[lo] == id;
}

template <bool EXCL>
__global__ void __launch_bounds__(kRedoThreads)
score_redo_kernel(const __nv_bfloat16* __restrict__ sess, const __nv_bfloat16* __restrict__ table, int64_t batch,
                  int64_t num_items, int dim, int k, int64_t id_base, const int32_t* __restrict__ redo,
                  float* __restrict__ top_val, int64_t* __restrict__ top_idx, const int64_t* __restrict__ targets,
                  int32_t* __restrict__ hit_pos, Exclusion excl) {
  extern __shared__ float redo_smem[];       // session row [dim], then lists, then (EXCL) the row's exclusion list
  // a small persistent grid; the flags of kRedoThreads rows are read at once, so rows that need no
  // recomputation (normally all of them) cost one coalesced load per 256 rows
  __shared__ int32_t s_flag[kRedoThreads];
  for (int64_t row0 = (int64_t)blockIdx.x * kRedoThreads; row0 < batch; row0 += (int64_t)gridDim.x * kRedoThreads) {
  const int32_t mine = row0 + threadIdx.x < batch ? redo[row0 + threadIdx.x] : 0;
  if (__syncthreads_or(mine) == 0) continue;  // CTA-uniform
  s_flag[threadIdx.x] = mine;
  __syncthreads();
  for (int rr = 0; rr < kRedoThreads; ++rr) {
  if (s_flag[rr] == 0) continue;              // CTA-uniform
  const int64_t row = row0 + rr;
  __syncthreads();                           // the previous row's lists are no longer read
  float* s_row = redo_smem;
  float* l_val = redo_smem + dim;            // [kRedoThreads][k]
  int32_t* l_idx = reinterpret_cast<int32_t*>(l_val + kRedoThreads * k);
  for (int d = threadIdx.x; d < dim; d += kRedoThreads) s_row[d] = __bfloat162float(sess[row * dim + d]);
  float* mv = l_val + threadIdx.x * k;
  int32_t* mi = l_idx + threadIdx.x * k;
  for (int t = 0; t < k; ++t) { mv[t] = -INFINITY; mi[t] = INT32_MAX; }
  int64_t* s_excl = reinterpret_cast<int64_t*>(l_idx + kRedoThreads * k);   // 8-byte aligned: dim % 64 == 0
  if (EXCL)
    for (int64_t i = threadIdx.x; i < excl.width; i += kRedoThreads) s_excl[i] = excl.ids[row * excl.width + i];
  __syncthreads();
  for (int64_t item = threadIdx.x; item < num_items; item += kRedoThreads) {
    const __nv_bfloat16* e = table + item * dim;
    float acc = 0.f;
    for (int d = 0; d < dim; d += 2) {
      const float2 p = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(e + d));
      acc = fmaf(s_row[d], p.x, acc);
      acc = fmaf(s_row[d + 1], p.y, acc);
    }
    if (acc > mv[k - 1] && !(EXCL && listed(s_excl, (int)excl.width, id_base + item))) {
      // ascending ids per thread: strict '>' keeps the lower id
      int t = k - 1;
      while (t > 0 && mv[t - 1] < acc) { mv[t] = mv[t - 1]; mi[t] = mi[t - 1]; --t; }
      mv[t] = acc;
      mi[t] = (int32_t)item;
    }
  }
  __syncthreads();
  // k selection passes over the kRedoThreads*k candidates by (score desc, id asc)
  __shared__ float r_val[kRedoThreads / 32];
  __shared__ int32_t r_idx[kRedoThreads / 32];
  float prev_v = INFINITY;
  int32_t prev_i = -1;
  int found = -1;
  for (int t = 0; t < k; ++t) {
    float bv = -INFINITY;
    int32_t bi = INT32_MAX;
    for (int c = threadIdx.x; c < kRedoThreads * k; c += kRedoThreads) {
      const float v = l_val[c];
      const int32_t i = l_idx[c];
      const bool after_prev = v < prev_v || (v == prev_v && i > prev_i);
      if (after_prev && (v > bv || (v == bv && i < bi))) { bv = v; bi = i; }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
      const int32_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if ((threadIdx.x & 31) == 0) { r_val[threadIdx.x >> 5] = bv; r_idx[threadIdx.x >> 5] = bi; }
    __syncthreads();
    bv = r_val[0]; bi = r_idx[0];
    for (int q = 1; q < kRedoThreads / 32; ++q)
      if (r_val[q] > bv || (r_val[q] == bv && r_idx[q] < bi)) { bv = r_val[q]; bi = r_idx[q]; }
    if (threadIdx.x == 0) {
      top_val[row * k + t] = bv;
      top_idx[row * k + t] = bi == INT32_MAX ? INT64_MAX : id_base + bi;
      if (targets != nullptr && found < 0 && bi != INT32_MAX && id_base + bi == targets[row]) found = t;
    }
    prev_v = bv;
    prev_i = bi;
    __syncthreads();
  }
  if (threadIdx.x == 0 && targets != nullptr) hit_pos[row] = found;
  }
  __syncthreads();                           // s_flag is rewritten by the next block of rows
  }
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n4) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = ldg4(src + 4 * i);
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 packed;
    packed.x = *reinterpret_cast<uint32_t*>(&lo);
    packed.y = *reinterpret_cast<uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(dst + 4 * i) = packed;
  }
}

struct TcPlan {
  Schedule sch;
  int grid;
  int cap, cap_sub;
  int col_parts;   // epilogue warps per TMEM lane quarter: 2 (default) or 4
  bool pairs;   // CTA pairs (cta_group::2): a row tile is 256 rows, grid = 2 x units, workers = 74 SM pairs
};

bool use_cta_pairs() {
  static const bool on = [] {
    const char* e = getenv("ETPGT_SCORE_2CTA");   // comparison knob: 0 = one CTA per unit (round 1's kernel shape)
    return e == nullptr || atoi(e) != 0;
  }();
  return on;
}

int epilogue_col_parts() {
  static const int parts = [] {
    // two epilogue warps per lane quarter; 4 (comparison knob) was measured slower: 350 instead of 215 dumped pieces
    // per row (four lists over a quarter of the pieces each) and 0.93 instead of 0.75 ms
    const char* e = getenv("ETPGT_SCORE_EPI");
    return e != nullptr && atoi(e) == 4 ? 4 : 2;
  }();
  return parts;
}

TcPlan tc_plan(int64_t batch, int64_t num_items, int k) {
  TcPlan p;
  p.pairs = use_cta_pairs();
  p.col_parts = epilogue_col_parts();
  const int unit_rows = p.pairs ? 2 * BLOCK_M : BLOCK_M;
  const int workers = p.pairs ? kNumSMs / 2 : kNumSMs;
  const int m_tiles = (int)((batch + unit_rows - 1) / unit_rows);
  const int total_tiles = (int)((num_items + BLOCK_N - 1) / BLOCK_N);
  // tail ranges stay >= 64 tiles (512 chunks) so that every range's own threshold is tight enough for
  // the select kernel's survivor buffer
  int max_splits = total_tiles / 64 > 1 ? total_tiles / 64 : 1;
  if (max_splits > 32) max_splits = 32;
  const int max_forced = total_tiles / 32 > 1 ? (total_tiles / 32 > 32 ? 32 : total_tiles / 32) : 1;   // tuning knob only
  const int m_full = (m_tiles / workers) * workers;   // whole waves: one full-catalogue unit per row tile
  const int tail = m_tiles - m_full;
  int splits = 1;
  if (tail > 0) {
    // cost model fitted on B200: time ~ waves * (range length + a warm-up worth ~half a full range)
    double best_cost = 1e30;
    for (int s = 1; s <= max_splits; ++s) {
      const int per = (total_tiles + s - 1) / s;
      const int real = (total_tiles + per - 1) / per;
      const int waves = (real * tail + workers - 1) / workers;
      const double cost = (double)waves * ((double)per / (double)total_tiles + 0.5);
      if (cost < best_cost - 1e-9) { best_cost = cost; splits = s; }
    }
    if (const char* forced = getenv("ETPGT_SCORE_SPLITS")) {  // tuning knob
      const int f = atoi(forced);
      if (f >= 1 && f <= max_forced) splits = f;
    }
  }
  p.sch.unit_rows = unit_rows;
  p.sch.m_full = m_full;
  p.sch.total_tiles = total_tiles;
  p.sch.tiles_per_split = (total_tiles + splits - 1) / splits;
  p.sch.tail_splits = (total_tiles + p.sch.tiles_per_split - 1) / p.sch.tiles_per_split;
  p.grid = (m_full + tail * p.sch.tail_splits) * (p.pairs ? 2 : 1);
  // slots per (row, range): every column part keeps its own list over its share of the pieces, so
  // ~ P*K*(1 + ln(pieces/(P*K))) pieces are expected (+ ~25 % from the lockstep merges); 1.6x head-room (sized
  // for the longest range), overflow is handled exactly by the fallback kernel
  const double chunks = (double)(m_full > 0 ? total_tiles : p.sch.tiles_per_split) * (BLOCK_N / DUMPW);
  const int kc = k <= 10 ? 10 : k <= 20 ? 20 : 32;
  const double lists = (double)p.col_parts * kc;
  double expect = lists * (1.0 + (chunks > lists ? log(chunks / lists) : 0.0));
  int cap = (int)(1.6 * expect) + 16;
  if (cap > (int)chunks) cap = (int)chunks;
  if (const char* forced = getenv("ETPGT_SCORE_CAP")) {  // test hook: force slot-buffer overflow
    const int f = atoi(forced);
    if (f >= 1) cap = f;
  }
  const int subs = p.col_parts / 2;
  p.cap_sub = (cap + subs - 1) / subs < 1 ? 1 : (cap + subs - 1) / subs;
  p.cap = p.cap_sub * subs;
  return p;
}

size_t tc_smem_bytes(int num_kb, int stages, bool pairs) {
  return 1024 + (size_t)num_kb * A_KBLOCK_BYTES + (size_t)stages * (pairs ? B_STAGE_BYTES / 2 : B_STAGE_BYTES) +
         sizeof(RowShared) + sizeof(Barriers) + 64;
}

}  // namespace
}  // namespace etpgt

using namespace etpgt;

extern "C" int etpgt_f32_to_bf16(const float* src, void* dst, int64_t n, etpgt_stream_t stream) {
  ETPGT_REQUIRE(n >= 0 && n % 4 == 0, "f32_to_bf16: element count must be a multiple of 4");
  if (n == 0) return ETPGT_OK;
  f32_to_bf16_kernel<<<grid_for(n / 4, 256 * 4, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src, static_cast<__nv_bfloat16*>(dst), n / 4);
  ETPGT_CHECK_LAUNCH("f32_to_bf16");
  return ETPGT_OK;
}

extern "C" size_t etpgt_score_topk_bf16_workspace_bytes(int64_t batch, int64_t num_items, int k) {
  if (batch <= 0 || num_items <= 0 || k <= 0) return 256;
  const TcPlan p = tc_plan(batch, num_items, k);
  const size_t units = (size_t)p.sch.num_parts(batch);
  return align_up(units * p.cap * DUMPW * sizeof(float)) + align_up(units * p.cap * sizeof(int2)) +
         2 * align_up(kMaxColParts * units * sizeof(float)) + 2 * align_up((size_t)batch * sizeof(int32_t)) + 256;
}

namespace {

// The scorer behind etpgt_score_topk_bf16_eval (excl.ids == nullptr) and etpgt_score_topk_bf16_exclude (k_any: k may
// exceed the eligible items, whose missing slots become (-inf, INT64_MAX) sentinels).
int score_topk_bf16_run(const void* sess_bf16, const void* table_bf16, int64_t batch, int64_t num_items, int dim,
                        int k, int64_t id_base, float* top_val, int64_t* top_idx, const int64_t* targets,
                        int32_t* hit_pos, Exclusion excl, bool k_any, void* ws, size_t ws_bytes,
                        etpgt_stream_t stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const bool use_excl = excl.ids != nullptr;
  ETPGT_REQUIRE((targets == nullptr) == (hit_pos == nullptr), "score_topk_bf16: targets and hit_pos come together");
  ETPGT_REQUIRE(dim == 64 || dim == 128 || dim == 192 || dim == 256,
                "score_topk_bf16: dim %d must be a multiple of 64 up to 256", dim);
  ETPGT_REQUIRE(batch >= 0 && num_items >= 1 && num_items < (int64_t(1) << 31), "score_topk_bf16: bad sizes");
  if (k_any) {
    ETPGT_REQUIRE(k >= 1 && k <= kMaxKTc, "score_topk_bf16: k=%d must be in [1, %d]", k, kMaxKTc);
  } else {
    ETPGT_REQUIRE(k >= 1 && k <= kMaxKTc && k <= num_items, "score_topk_bf16: k=%d must be in [1, min(%d, num_items)]",
                  k, kMaxKTc);
  }
  ETPGT_REQUIRE(((uintptr_t)sess_bf16 & 15) == 0 && ((uintptr_t)table_bf16 & 15) == 0,
                "score_topk_bf16: operands must be 16-byte aligned");
  if (ws_bytes < etpgt_score_topk_bf16_workspace_bytes(batch, num_items, k)) {
    set_error("score_topk_bf16: workspace too small");
    return ETPGT_EWORKSPACE;
  }
  if (batch == 0) return ETPGT_OK;
  const TcPlan p = tc_plan(batch, num_items, k);
  // the exclusion variant exists for the default kernel shape only (CTA pairs, two column parts)
  ETPGT_REQUIRE(!use_excl || (p.pairs && p.col_parts == 2),
                "score_topk_bf16_exclude: exclusion needs the default scorer configuration (unset ETPGT_SCORE_2CTA and "
                "ETPGT_SCORE_EPI)");
  Workspace w(ws, ws_bytes);
  const size_t units = (size_t)p.sch.num_parts(batch);
  DumpBuffers dump;
  dump.scores = w.take<float>(units * p.cap * DUMPW);
  dump.meta = w.take<int2>(units * p.cap);
  dump.count = w.take<int32_t>(kMaxColParts * units);
  dump.threshold = w.take<float>(kMaxColParts * units);
  dump.units = (int64_t)units;
  dump.cap = p.cap;
  dump.cap_sub = p.cap_sub;
  dump.col_parts = p.col_parts;
  int32_t* redo = w.take<int32_t>(batch);
  CUtensorMap map_sess, map_items;
  if (!make_map_bf16(&map_sess, sess_bf16, batch, dim, dim, BLOCK_M) ||
      !make_map_bf16(&map_items, table_bf16, num_items, dim, dim, p.pairs ? BLOCK_N / 2 : BLOCK_N)) {
    set_error("score_topk_bf16: cuTensorMapEncodeTiled failed");
    return ETPGT_ECUDA;
  }
  const int num_kb = dim / BLOCK_K;
  const int stages = p.pairs ? kMaxStages : kMaxStages / 2;
  int pending_merge = kDefaultPendingMerge;
  if (const char* forced = getenv("ETPGT_SCORE_PENDING")) {  // tuning knob
    const int f = atoi(forced);
    if (f >= 1 && f <= kPendingMerge + 1 - BLOCK_N / 2 / DUMPW) pending_merge = f;
  }
  // the exclusion variant keeps its epilogue threads' cursors behind the barriers
  const size_t smem = tc_smem_bytes(num_kb, stages, p.pairs) + (use_excl ? 4 * 2 * 32 * sizeof(ExclCursor) : 0);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(p.grid);
  cfg.blockDim = dim3(threads_for(p.col_parts));
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.pairs ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
#define LAUNCH4(NKB, KC, PR, CP_, EX)                                                                              \
  {                                                                                                                \
    cudaFuncSetAttribute(score_dump_tc_kernel<NKB, KC, PR, CP_, EX>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                         (int)smem);                                                                               \
    cudaLaunchKernelEx(&cfg, score_dump_tc_kernel<NKB, KC, PR, CP_, EX>, map_sess, map_items, batch, num_items,    \
                       stages, p.sch, dump, pending_merge, excl);                                                  \
  }
#define LAUNCH3(NKB, KC, PR)                           \
  {                                                    \
    if (p.col_parts == 4) LAUNCH4(NKB, KC, PR, 4, false) \
    else LAUNCH4(NKB, KC, PR, 2, false)                \
  }
#define LAUNCH2(NKB, KC)                            \
  {                                                 \
    if (use_excl) LAUNCH4(NKB, KC, true, 2, true)   \
    else if (p.pairs) LAUNCH3(NKB, KC, true)        \
    else LAUNCH3(NKB, KC, false)                    \
  }
#define LAUNCH(NKB)                    \
  {                                    \
    if (k <= 10) LAUNCH2(NKB, 10)      \
    else if (k <= 20) LAUNCH2(NKB, 20) \
    else LAUNCH2(NKB, 32)              \
  }
  const bool stats = getenv("ETPGT_SCORE_STATS") != nullptr;   // tuning aid (synchronises)
  cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
  if (stats) {
    for (auto& e : ev) cudaEventCreate(&e);
    cudaEventRecord(ev[0], stream);
  }
  switch (num_kb) {
    case 1: LAUNCH(1) break;
    case 2: LAUNCH(2) break;
    case 3: LAUNCH(3) break;
    default: LAUNCH(4) break;
  }
#undef LAUNCH
#undef LAUNCH2
#undef LAUNCH3
#undef LAUNCH4
  ETPGT_CHECK_LAUNCH("score_dump_tc");
  if (stats) cudaEventRecord(ev[1], stream);
  score_select_kernel<<<(unsigned)((batch + kSelectWarps - 1) / kSelectWarps), kSelectWarps * 32, 0, stream>>>(
      dump, batch, p.sch, k, id_base, top_val, top_idx, redo, targets, hit_pos);
  ETPGT_CHECK_LAUNCH("score_select");
  if (stats) cudaEventRecord(ev[2], stream);
  const size_t redo_smem = ((size_t)dim + (size_t)kRedoThreads * k * 2) * sizeof(float) +
                           (use_excl ? (size_t)excl.width * sizeof(int64_t) : 0);
  const int64_t redo_blocks = (batch + kRedoThreads - 1) / kRedoThreads;
  const unsigned redo_grid = (unsigned)(redo_blocks < 2 * kNumSMs ? redo_blocks : 2 * kNumSMs);
  if (use_excl) {
    if (redo_smem > 48 * 1024)
      cudaFuncSetAttribute(score_redo_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)redo_smem);
    score_redo_kernel<true><<<redo_grid, kRedoThreads, redo_smem, stream>>>(
        static_cast<const __nv_bfloat16*>(sess_bf16), static_cast<const __nv_bfloat16*>(table_bf16), batch,
        num_items, dim, k, id_base, redo, top_val, top_idx, targets, hit_pos, excl);
  } else {
    if (redo_smem > 48 * 1024)
      cudaFuncSetAttribute(score_redo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)redo_smem);
    score_redo_kernel<false><<<redo_grid, kRedoThreads, redo_smem, stream>>>(
        static_cast<const __nv_bfloat16*>(sess_bf16), static_cast<const __nv_bfloat16*>(table_bf16), batch,
        num_items, dim, k, id_base, redo, top_val, top_idx, targets, hit_pos, excl);
  }
  ETPGT_CHECK_LAUNCH("score_redo");
  if (stats) {   // dump volume, fallback rows, kernel times
    std::vector<int32_t> h_redo(batch), h_count(kMaxColParts * units);
    cudaStreamSynchronize(stream);
    float ms_dump = 0.f, ms_select = 0.f;
    cudaEventElapsedTime(&ms_dump, ev[0], ev[1]);
    cudaEventElapsedTime(&ms_select, ev[1], ev[2]);
    for (auto& e : ev) cudaEventDestroy(e);
    fprintf(stderr, "score_topk_bf16: dump %.3f ms, select %.3f ms\n", ms_dump, ms_select);
    cudaMemcpy(h_redo.data(), redo, batch * sizeof(int32_t), cudaMemcpyDeviceToHost);
    cudaMemcpy(h_count.data(), dump.count, kMaxColParts * units * sizeof(int32_t), cudaMemcpyDeviceToHost);
    int64_t redo_rows = 0, pieces = 0, worst = 0;
    for (int64_t i = 0; i < batch; ++i) redo_rows += h_redo[i];
    for (size_t i = 0; i < units; ++i) {
      int64_t c = 0;
      for (int cp = 0; cp < p.col_parts; ++cp) c += h_count[(size_t)cp * units + i];
      pieces += c;
      worst = c > worst ? c : worst;
    }
    fprintf(stderr, "score_topk_bf16: grid %d, %zu (row, range) units, cap %d, %.1f pieces per unit (max %lld), %lld rows recomputed\n",
            p.grid, units, p.cap, (double)pieces / (double)units, (long long)worst, (long long)redo_rows);
  }
  return ETPGT_OK;
}

}  // namespace

extern "C" int etpgt_score_topk_bf16_eval(const void* sess_bf16, const void* table_bf16, int64_t batch,
                                          int64_t num_items, int dim, int k, int64_t id_base, float* top_val,
                                          int64_t* top_idx, const int64_t* targets, int32_t* hit_pos, void* ws,
                                          size_t ws_bytes, etpgt_stream_t stream) {
  return score_topk_bf16_run(sess_bf16, table_bf16, batch, num_items, dim, k, id_base, top_val, top_idx, targets,
                             hit_pos, Exclusion{nullptr, 0, 0}, false, ws, ws_bytes, stream);
}

extern "C" int etpgt_score_topk_bf16_exclude(const void* sess_bf16, const void* table_bf16, int64_t batch,
                                             int64_t num_items, int dim, int k, int64_t id_base, float* top_val,
                                             int64_t* top_idx, const int64_t* targets, int32_t* hit_pos,
                                             const int64_t* exclude, int64_t exclude_width, void* ws, size_t ws_bytes,
                                             etpgt_stream_t stream) {
  ETPGT_REQUIRE(exclude_width >= 0 && exclude_width <= kMaxExcludeWidth,
                "score_topk_bf16_exclude: exclude_width %lld must be in [0, %lld]", (long long)exclude_width,
                (long long)kMaxExcludeWidth);
  ETPGT_REQUIRE(exclude_width == 0 || batch == 0 || exclude != nullptr, "score_topk_bf16_exclude: null exclude list");
  // width 0: nothing to exclude, the unfiltered kernels run (k > num_items still yields sentinels)
  const Exclusion excl{exclude_width > 0 ? exclude : nullptr, exclude_width, id_base};
  return score_topk_bf16_run(sess_bf16, table_bf16, batch, num_items, dim, k, id_base, top_val, top_idx, targets,
                             hit_pos, excl, true, ws, ws_bytes, stream);
}

extern "C" int etpgt_score_topk_bf16(const void* sess_bf16, const void* table_bf16, int64_t batch,
                                     int64_t num_items, int dim, int k, int64_t id_base, float* top_val,
                                     int64_t* top_idx, void* ws, size_t ws_bytes, etpgt_stream_t stream) {
  return etpgt_score_topk_bf16_eval(sess_bf16, table_bf16, batch, num_items, dim, k, id_base, top_val, top_idx, nullptr,
                                    nullptr, ws, ws_bytes, stream);
}
