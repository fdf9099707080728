/* etpgt_b200 — C ABI of the B200-native hot path of the `etpgt` session recommender.
 *
 * The reference (Axionis47/GAT-Recommendation) is pure Python and has no FFI; its drop-in
 * boundary is the Python module API of etpgt/model, etpgt/train/losses.py and
 * etpgt/utils/metrics.py (SURVEY.md §8b).  These are the entry points a binding for that
 * path uses; each one names the reference code it replaces.  INTEGRATION.md shows the
 * ctypes stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless it says "host";
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never
 *     allocates and never synchronises; scratch comes from `ws` sized by *_workspace_bytes;
 *   - returns 0, or a negative ETPGT_E* code with a thread-local message in
 *     etpgt_last_error(); nothing is launched when an argument check fails;
 *   - API-side indices are int64 (the reference's dtype); internal structures are int32;
 *   - feature matrices are fp32 row-major with D in {32,64,128,256};
 *   - no global mutable state, re-entrant, no CPU fallback anywhere.
 */
#ifndef ETPGT_B200_H
#define ETPGT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ETPGT_OK 0
#define ETPGT_EINVAL (-1)   /* bad argument / unsupported shape */
#define ETPGT_ECUDA (-2)    /* CUDA runtime error at launch */
#define ETPGT_EWORKSPACE (-3) /* workspace too small */

typedef void* etpgt_stream_t; /* cudaStream_t */

int etpgt_version(void);
const char* etpgt_last_error(void);
/* number of kernel launches issued by this library (all threads of the process; autograd runs
 * backward on worker threads) since the last reset — bench.py's `gpu_launches`. */
int64_t etpgt_launch_count(void);
void etpgt_reset_launch_count(void);

/* ---- index structures ------------------------------------------------------------------
 * Destination-sorted CSR and source-sorted CSC of an edge list, both stable (ties keep the
 * original edge order).  Replaces the COO scatter inside PyG's MessagePassing.propagate that
 * etpgt/model/graph_transformer.py:174, gat.py:137 and graphsage.py:75 reach.
 *   rowptr[N+1], col[E] (source of the p-th CSR edge), eperm[E] (its original index),
 *   colptr[N+1], row[E] (destination of the p-th CSC edge), cpos[E] (its CSR position). */
size_t etpgt_csr_workspace_bytes(int64_t num_edges, int64_t num_nodes);
int etpgt_csr_from_coo(const int64_t* src, const int64_t* dst, int64_t num_edges, int64_t num_nodes,
                       int32_t* rowptr, int32_t* col, int32_t* eperm,
                       int32_t* colptr, int32_t* row, int32_t* cpos,
                       void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* ptr[S+1] from a non-decreasing segment-id vector (PyG `batch`): etpgt/model/base.py:146-155. */
int etpgt_segment_ptr(const int64_t* seg_ids, int64_t n, int64_t num_segments, int32_t* ptr,
                      etpgt_stream_t stream);

/* ---- a1-a3: per-batch session subgraphs and negatives on the device ------------------------
 * Replaces SessionDataset._build_session_subgraph / collate_fn / _sample_negatives
 * (etpgt/train/dataloader.py:107-202) and create_batch_from_sessions' edge rules
 * (scripts/pipeline/run_full_pipeline.py:120-166).
 *
 * item_graph_build (one-off): lookup structure over the stored edge list (item_i[e], item_j[e]) in
 * its stored order: gptr[num_items+1] rows keyed by item_i, gcol[E] = item_j sorted inside a row,
 * gidx[E] = stored row index of that edge. */
size_t etpgt_item_graph_workspace_bytes(int64_t num_edges);
int etpgt_item_graph_build(const int64_t* item_i, const int64_t* item_j, int64_t num_edges,
                           int64_t num_items, int32_t* gptr, int32_t* gcol, int32_t* gidx,
                           void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* Sessions are sess_items[sess_ptr[s] : sess_ptr[s+1]] in chronological order (target = last
 * event).  Only the last max_len events are used (max_len <= 65); context = all but the last;
 * nodes = sorted unique context items; an edge of the stored list is kept iff both ends are context
 * items, in stored order and direction.  session_ids [S] (or NULL = 0..S-1) selects the batch's
 * sessions out of the resident store.  symmetrize appends the reversed copies after the forward
 * ones; self_loop_if_empty adds one loop per node when no edge was kept.
 * count: node_ptr / edge_ptr [S+1] (exclusive prefix sums; the caller reads the two totals to size
 * the outputs).  fill: x [N] item ids, batch [N] session index, edge_src / edge_dst [E] with the
 * cumulative node offset added (PyG collate layout), target [S]. */
size_t etpgt_session_subgraphs_workspace_bytes(int64_t num_sessions, int64_t num_edges);
int etpgt_session_subgraphs_count(const int32_t* gptr, const int32_t* gcol, const int64_t* sess_ptr,
                                  const int64_t* sess_items, const int64_t* session_ids,
                                  int64_t num_sessions, int max_len,
                                  int symmetrize, int self_loop_if_empty,
                                  int32_t* node_ptr, int32_t* edge_ptr,
                                  void* ws, size_t ws_bytes, etpgt_stream_t stream);
int etpgt_session_subgraphs_fill(const int32_t* gptr, const int32_t* gcol, const int32_t* gidx,
                                 const int64_t* sess_ptr, const int64_t* sess_items,
                                 const int64_t* session_ids, int64_t num_sessions, int max_len,
                                 int symmetrize,
                                 int self_loop_if_empty, const int32_t* node_ptr,
                                 const int32_t* edge_ptr, int64_t num_edges,
                                 int64_t* x, int64_t* batch, int64_t* edge_src, int64_t* edge_dst,
                                 int64_t* target, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* out[s, slot] = uniform id in [1, num_items) that is not among the last max_len events of session
 * s (duplicates between slots allowed).  Philox4x32-10, key = seed, counter = (GLOBAL session index
 * = session_ids[s], or session_base + s when session_ids is NULL; slot, attempt / 4, step), word attempt % 4, candidate = 1 + ((word * (num_items-1)) >> 32):
 * identical for any partition of the sessions over GPUs. */
int etpgt_sample_negatives(uint64_t seed, uint32_t step, int64_t session_base,
                           const int64_t* sess_ptr, const int64_t* sess_items,
                           const int64_t* session_ids, int64_t num_sessions,
                           int max_len, int64_t num_items, int num_neg, int64_t* out,
                           etpgt_stream_t stream);
/* Shared negative pool for the sampled softmax (etpgt_pool_softmax_*): num_sampled item ids drawn with replacement
 * from q(i) = w_i / W, cum [num_items + 1] = (0, w_0, w_0 + w_1, ..., W) on the device, 0 < W < 2^62.  Draw j:
 * Philox4x32-10, key (seed lo, seed hi), counter (j >> 1, 0x504F4F4C, 0, step), u = c[2(j&1)] | c[2(j&1)+1] << 32,
 * r = umulhi64(u, W), the id i with cum[i] <= r < cum[i+1] (zero-weight ids are never drawn).  pool_ids [num_sampled]
 * is written sorted ascending, log_q [num_sampled] = (float) log(num_sampled * w_id / W) in fp64.  Depends on
 * (seed, step) only: every data-parallel rank draws the same pool.  No allocation, no synchronisation. */
size_t etpgt_sample_item_pool_workspace_bytes(int64_t num_sampled);
int etpgt_sample_item_pool(const int64_t* cum, int64_t num_items, int64_t num_sampled, uint64_t seed, uint32_t step,
                           int64_t* pool_ids, float* log_q, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* In-batch negatives for etpgt_pool_softmax_*: the column list of the batch's targets [batch] (one column per
 * session) merged with the optional sorted pool pool_ids / pool_log_q [num_pool] of etpgt_sample_item_pool
 * (num_pool = 0: no pool, both may be NULL).  columns [num_pool + batch] is written ascending; among equal ids the pool
 * entries come first, then the in-batch entries in session order.  A pool entry keeps its log_q.  First the streaming
 * estimate of each item's share of the targets is updated: for each distinct target i in [0, num_items), i !=
 * padding_idx, with n copies among the batch,
 *   freq[i] = freq[i] * (1 - decay)^(step - last[i]) + decay * n / batch,   last[i] = step
 * (freq fp64 [num_items], last int64 [num_items]; steps increase from call to call).  The in-batch column of session
 * b then gets log_q = (float) log(batch * freq[t_b]) in fp64, read after the update.  A target outside
 * [0, num_items) never touches freq / last; its column, and that of a padding target, gets log_q = +inf (never a
 * negative).  decay in (0, 1], step >= 0.  Deterministic, no allocation, no synchronisation, graph-capturable. */
size_t etpgt_in_batch_columns_workspace_bytes(int64_t batch, int64_t num_pool);
int etpgt_in_batch_columns(const int64_t* targets, int64_t batch, const int64_t* pool_ids, const float* pool_log_q,
                           int64_t num_pool, double* freq, int64_t* last, int64_t num_items, int64_t padding_idx,
                           int64_t step, double decay, int64_t* columns, float* log_q, void* ws, size_t ws_bytes,
                           etpgt_stream_t stream);

/* ---- a4: item embedding + Laplacian-PE projection -------------------------------------
 * out[n] = table[ids[n]] (+ pe[pe_row(n)] @ w_pe^T + b_pe);  pe_row(n) = n when
 * pe_per_node else ids[n].  etpgt/model/graph_transformer.py:140-152,
 * etpgt/encodings/laplacian_pe.py:170-199.  pe == NULL skips the projection. */
int etpgt_embed_pe_fwd(const int64_t* ids, int64_t n, const float* table, int64_t num_items,
                       const float* pe, int pe_per_node, const float* w_pe, const float* b_pe,
                       int k_pe, int dim, float* out, etpgt_stream_t stream);
/* The same, also writing out split as bf16 pairs out = out_hi + out_lo (hi = bf16(x), lo = bf16(x - hi), exactly
 * what etpgt_split_bf16 produces): the operand format of the first layer's tensor-core projection, so that
 * layer needs no split pass.  out_hi / out_lo [n, dim] bf16, both or neither. */
int etpgt_embed_pe_fwd_split(const int64_t* ids, int64_t n, const float* table, int64_t num_items,
                             const float* pe, int pe_per_node, const float* w_pe, const float* b_pe,
                             int k_pe, int dim, float* out, void* out_hi, void* out_lo, etpgt_stream_t stream);
/* Deterministic backward: d_table (dense [num_items, dim], caller-zeroed, rows are ADDED),
 * d_w_pe [dim,k_pe], d_b_pe [dim] (overwritten; NULL when pe == NULL).  Row padding_idx
 * (etpgt/model/base.py:36; -1 = none) receives no gradient. */
size_t etpgt_embed_pe_bwd_workspace_bytes(int64_t n, int dim, int k_pe);
int etpgt_embed_pe_bwd(const int64_t* ids, int64_t n, const float* d_out, int64_t num_items,
                       const float* pe, int pe_per_node, int k_pe, int dim, int64_t padding_idx,
                       float* d_table, float* d_w_pe, float* d_b_pe,
                       void* ws, size_t ws_bytes, etpgt_stream_t stream);

/* ---- a5: fused TransformerConv ----------------------------------------------------------
 * qkvs [N, 4*dim] = (query | key | value | skip) projections of x (one GEMM by the caller).
 * Per destination i and head h: a_e = <q_i,k_j>/sqrt(C); alpha = exp(a_e-m_i)/(sum+1e-16);
 * agg_i = sum alpha*mask_e*v_j; beta = sigmoid(w_beta . [agg, s, agg-s]); out = beta*s+(1-beta)*agg.
 * PyG TransformerConv(concat=True, beta=True) as used at graph_transformer.py:73-98,174.
 * alpha_mask [E, heads] in ORIGINAL edge order (dropout mask already scaled) or NULL.
 * w_beta == NULL selects beta=False (out = agg + s).
 * Saved for backward: agg [N,dim], beta [N], m [N,heads], inv_l [N,heads]. */
int etpgt_tconv_fwd(const float* qkvs, int64_t num_nodes, int dim, int heads,
                    const int32_t* rowptr, const int32_t* col, const int32_t* eperm, int64_t num_edges,
                    const float* w_beta, const float* alpha_mask,
                    float* out, float* agg, float* beta, float* m, float* inv_l,
                    etpgt_stream_t stream);
/* Backward, no atomics: a destination pass (d_query, d_skip, per-edge coefficients) then a
 * source pass over the CSC (d_key, d_value).  d_qkvs [N,4*dim] is overwritten; d_w_beta [3*dim]
 * overwritten (NULL when w_beta == NULL). */
/* Hub rows.  A destination (forward, backward destination pass) or source (backward source pass) with more than
 * 256 edges is cut into chunks of 256 edges; one CTA per chunk stages the row's query (and d_agg) in shared memory,
 * its lane groups each walk a slice, and the (m, l, acc) / gradient partials are combined in a fixed order inside
 * the CTA and then over the chunks of the row — no atomics, bit-reproducible (north_star (2): "shared-memory staging
 * of hub-node rows"; the reference's generator is zipf(1.5), scripts/data/00_generate_synthetic_data.py:53).
 * etpgt_hub_plan builds the row / chunk lists for the CSR (rowptr) and CSC (colptr) sides once per graph index,
 * deterministically (prefix sums); plan[0..3] (int32, device) = #hub destinations, #their chunks, #hub sources,
 * #their chunks.  The *_hub entry points take the plan (NULL = the plain row kernels) and a workspace for the
 * per-chunk partials; rows at or below the threshold run in the row kernels as before. */
size_t etpgt_hub_plan_bytes(int64_t num_edges);
size_t etpgt_hub_plan_workspace_bytes(int64_t num_nodes);
int etpgt_hub_plan(const int32_t* rowptr, const int32_t* colptr, int64_t num_nodes, int64_t num_edges, void* plan,
                   void* ws, size_t ws_bytes, etpgt_stream_t stream);
size_t etpgt_tconv_hub_workspace_bytes(int64_t num_edges, int dim);
int etpgt_tconv_fwd_hub(const float* qkvs, int64_t num_nodes, int dim, int heads, const int32_t* rowptr,
                        const int32_t* col, const int32_t* eperm, int64_t num_edges, const float* w_beta,
                        const float* alpha_mask, float* out, float* agg, float* beta, float* m, float* inv_l,
                        const void* hub_plan, void* hub_ws, size_t hub_ws_bytes, etpgt_stream_t stream);
/* The forward that also takes the BatchNorm statistics of its output while the rows are in registers
 * (graph_transformer.py:174-175: conv -> BatchNorm1d): bn_sums [2*dim] doubles = column sums of out and of out^2 over
 * all num_nodes rows — the input of etpgt_bn_finalize (append the row count for the data-parallel exchange) — so the
 * separate statistics pass of etpgt_bn_stats (one more read of [N, dim]) is not needed.  Persistent kernel, per-CTA
 * partial rows added in a fixed order: deterministic.  hub_plan may be NULL. */
size_t etpgt_tconv_fwd_bn_workspace_bytes(int dim);
int etpgt_tconv_fwd_bn(const float* qkvs, int64_t num_nodes, int dim, int heads, const int32_t* rowptr,
                       const int32_t* col, const int32_t* eperm, int64_t num_edges, const float* w_beta,
                       const float* alpha_mask, float* out, float* agg, float* beta, float* m, float* inv_l,
                       const void* hub_plan, void* hub_ws, size_t hub_ws_bytes, double* bn_sums, void* bn_ws,
                       size_t bn_ws_bytes, etpgt_stream_t stream);
int etpgt_tconv_bwd_split_hub(const float* qkvs, const float* d_out, int64_t num_nodes, int dim, int heads,
                              const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                              const int32_t* colptr, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                              const float* w_beta, const float* alpha_mask, const float* agg, const float* beta,
                              const float* m, const float* inv_l, float* d_qkvs, void* d_hi, void* d_lo,
                              float* d_colsum, float* d_w_beta, void* ws, size_t ws_bytes, const void* hub_plan,
                              void* hub_ws, size_t hub_ws_bytes, etpgt_stream_t stream);
size_t etpgt_tconv_bwd_workspace_bytes(int64_t num_nodes, int64_t num_edges, int dim, int heads);
int etpgt_tconv_bwd(const float* qkvs, const float* d_out, int64_t num_nodes, int dim, int heads,
                    const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                    const int32_t* colptr, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                    const float* w_beta, const float* alpha_mask,
                    const float* agg, const float* beta, const float* m, const float* inv_l,
                    float* d_qkvs, float* d_w_beta,
                    void* ws, size_t ws_bytes, etpgt_stream_t stream);

/* The same backward for the tensor-core projection path: instead of (or next to) the fp32 d_qkvs the
 * gradient rows are written already split as bf16 pairs d_hi + d_lo = d_qkvs (hi = bf16(x),
 * lo = bf16(x - hi), exactly what etpgt_split_bf16 would produce), and d_colsum [4*dim] receives the
 * column sums of d_qkvs (the gradient of the fused query|key|value|skip bias), reduced in a fixed
 * order.  d_qkvs may be NULL when d_hi / d_lo are given; d_colsum may be NULL. */
int etpgt_tconv_bwd_split(const float* qkvs, const float* d_out, int64_t num_nodes, int dim, int heads,
                          const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                          const int32_t* colptr, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                          const float* w_beta, const float* alpha_mask,
                          const float* agg, const float* beta, const float* m, const float* inv_l,
                          float* d_qkvs, void* d_hi, void* d_lo, float* d_colsum, float* d_w_beta,
                          void* ws, size_t ws_bytes, etpgt_stream_t stream);

/* ---- a5 (dense part): node projections on the tensor cores, fp32-grade ("split-bf16 x3") ----
 * Replaces the fp32 nn.Linear GEMMs of TransformerConv (lin_query/key/value/skip,
 * graph_transformer.py:73-98,174).  x = hi + lo with hi = bf16(x), lo = bf16(x - hi);
 * C = A_hi B_hi^T + A_hi B_lo^T + A_lo B_hi^T accumulated in fp32 in TMEM (tcgen05.mma), relative
 * error ~1e-5.  Operands are K-major bf16: A [M,K] (pitch lda), B [N,K] (pitch ldb), pitches
 * multiples of 8 elements; C fp32 [M,N] (pitch ldc); bias [N] or NULL.  a_lo == b_lo == NULL gives a
 * plain bf16 GEMM.  split_k: 1 = none, 0 = automatic (few output tiles, long K), >1 = forced; the
 * split-K partials are reduced in a fixed order (deterministic).
 *
 * split_bf16: src fp32 [rows, cols] (pitch ld_src) -> any of: hi/lo row-major [rows, cols] (pitch
 * ld_out), hi_t/lo_t transposed [cols, rows] (pitch ld_t), colsum [cols] (fp32 column sums). */
size_t etpgt_split_bf16_workspace_bytes(int64_t rows, int64_t cols);
int etpgt_split_bf16(const float* src, int64_t rows, int64_t cols, int64_t ld_src,
                     void* hi, void* lo, int64_t ld_out, void* hi_t, void* lo_t, int64_t ld_t,
                     float* colsum, void* ws, size_t ws_bytes, etpgt_stream_t stream);
size_t etpgt_gemm_bf16x3_workspace_bytes(int64_t m, int64_t n, int64_t k, int split_k);
int etpgt_gemm_bf16x3(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                      int64_t m, int64_t n, int64_t k, int64_t lda, int64_t ldb,
                      const float* bias, float* c, int64_t ldc, int split_k,
                      void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* The same with either operand stored MN-major, i.e. as the transpose: a_mn_major != 0 means A is
 * given as [K, M] row-major (pitch lda >= M), b_mn_major != 0 means B is given as [K, N] row-major
 * (pitch ldb >= N).  This is what the two backward GEMMs of a Linear layer need without any
 * transposed copies: dX[nodes,in] = dY[nodes,out] (K-major) x W[out,in] (B MN-major), and
 * dW[out,in] = dY[nodes,out] (A MN-major) x X[nodes,in] (B MN-major), K = nodes.
 * accumulate != 0: C += A B^T (+ bias) — the tiles are added to C by the TMA unit
 * (cp.reduce.async.bulk.tensor .add, one add per element: deterministic), which is how the residual
 * branch's gradient is merged into dX without a separate add pass. */
int etpgt_gemm_bf16x3_ex(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                         int64_t m, int64_t n, int64_t k, int64_t lda, int64_t ldb,
                         int a_mn_major, int b_mn_major,
                         const float* bias, int accumulate, float* c, int64_t ldc, int split_k,
                         void* ws, size_t ws_bytes, etpgt_stream_t stream);

/* ---- f4: the FFN variant's Linear -> GELU -> Dropout -> Linear -> Dropout (etpgt/model/graph_transformer.py:109-124,
 * 157-168, create_graph_transformer).  etpgt_gemm_bf16x3_gelu is etpgt_gemm_bf16x3 (K-major operands, no split-K)
 * whose epilogue has a second output: besides the fp32 pre-activation C = A B^T + bias (kept for the backward pass)
 * it writes h = dropout_p(gelu(C)) directly as the split-bf16 operand pair h_hi / h_lo [M, N] (pitch ldh) of the
 * second GEMM; the fp32 h and its split pass never exist.  GELU is nn.GELU()'s exact erf form; the mask is Philox
 * keyed by (seed, element), p = 0 disables it.  etpgt_gelu_bwd_split is the matching backward element pass:
 * du = d_h * mask * gelu'(u), written as the split-bf16 pair du_hi / du_lo [rows, cols] (pitch ld_out) with its
 * column sums (the first layer's bias gradient, NULL to skip; workspace = etpgt_split_bf16_workspace_bytes). */
int etpgt_gemm_bf16x3_gelu(const void* a_hi, const void* a_lo, const void* b_hi, const void* b_lo,
                           int64_t m, int64_t n, int64_t k, int64_t lda, int64_t ldb,
                           const float* bias, float* c, int64_t ldc,
                           void* h_hi, void* h_lo, int64_t ldh, double drop_p, uint64_t seed,
                           void* ws, size_t ws_bytes, etpgt_stream_t stream);
int etpgt_gelu_bwd_split(const float* d_h, const float* u, int64_t rows, int64_t cols, double drop_p, uint64_t seed,
                         void* du_hi, void* du_lo, int64_t ld_out, float* colsum,
                         void* ws, size_t ws_bytes, etpgt_stream_t stream);

/* ---- f4: Laplacian positional encoding on the device (etpgt/encodings/laplacian_pe.py:19-66: PyG
 * get_laplacian(normalization="sym") -> scipy eigsh(k+1, which="SM")).  The operator of the eigen solver
 * (etpgt_b200.encodings.laplacian_pe.compute_laplacian_pe(..., method="device"), Chebyshev-filtered subspace
 * iteration): y = alpha * (L x) + beta * x + gamma * z on a block of b <= 32 fp64 vectors stored [n, b] row-major,
 * L = I - D^-1/2 A D^-1/2 given by the graph's CSR rows (rowptr int64 [n+1], col int32, self loops removed,
 * parallel edges counted) and scale = deg^-1/2 (0 for isolated nodes).  z may be NULL; y must not alias x or z. */
int etpgt_lap_sym_block(const int64_t* rowptr, const int32_t* col, const double* scale, int64_t n, int b,
                        const double* x, const double* z, double alpha, double beta, double gamma,
                        double* y, etpgt_stream_t stream);

/* ---- a12: GAT edge-softmax aggregation and GraphSAGE mean aggregation ---------------------
 * PyG GATConv(add_self_loops=True) as used at etpgt/model/gat.py:49-109,137: h [N, width] with
 * width = heads*channels is the projected row, a_src/a_dst [N, heads] the attention scalars;
 * e = leaky_relu(a_src[j] + a_dst[i]); existing self loops are dropped and one self loop per node
 * is processed after the real edges; agg [N, width] = per-head sum alpha * h_j (the head mean /
 * concat + bias stay with the caller).  mask_edges [E, heads] (original edge order) and
 * mask_self [N, heads] are optional dropout masks (both or neither).  width in {32..1024}. */
int etpgt_gat_fwd(const float* h, const float* a_src, const float* a_dst, int64_t num_nodes, int width,
                  int heads, const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                  float negative_slope, const float* mask_edges, const float* mask_self,
                  float* agg, float* m, float* inv_l, etpgt_stream_t stream);
size_t etpgt_gat_bwd_workspace_bytes(int64_t num_nodes, int64_t num_edges, int heads);
int etpgt_gat_bwd(const float* h, const float* a_src, const float* a_dst, const float* d_agg,
                  const float* agg, int64_t num_nodes, int width, int heads,
                  const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                  const int32_t* colptr, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                  float negative_slope, const float* mask_edges, const float* mask_self,
                  const float* m, const float* inv_l, float* d_h, float* d_a_src, float* d_a_dst,
                  void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* concat=False (the reference's output layer and default, etpgt/model/gat.py:100-109) with the head mean inside the
 * edge kernels: etpgt_gat_fwd_mean also writes out_mean [N, channels] = mean over heads of agg + bias (agg is still
 * written: the backward pass reads it); needs etpgt_gat_mean_fused_supported(width, heads) != 0 (a head spans whole
 * lane-group rounds, e.g. channels a multiple of 128 at width >= 128).  etpgt_gat_bwd_mean takes EITHER d_agg
 * [N, heads*channels] or d_out_mean [N, channels] (the other NULL): with d_out_mean the per-head gradient
 * d_out / heads is expanded in registers — the [N, heads*channels] gradient never exists and the source pass
 * gathers channels*4 instead of heads*channels*4 bytes per edge.  The projection gradient goes EITHER to d_h (fp32)
 * or to d_h_hi / d_h_lo (split bf16, see etpgt_gat_input_scores_*). */
int etpgt_gat_mean_fused_supported(int width, int heads);
int etpgt_gat_fwd_mean(const float* h, const float* a_src, const float* a_dst, int64_t num_nodes, int width,
                       int heads, const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                       float negative_slope, const float* mask_edges, const float* mask_self, const float* bias,
                       float* agg, float* m, float* inv_l, float* out_mean, etpgt_stream_t stream);
int etpgt_gat_bwd_mean(const float* h, const float* a_src, const float* a_dst, const float* d_agg,
                       const float* d_out_mean, const float* agg, int64_t num_nodes, int width, int heads,
                       const int32_t* rowptr, const int32_t* col, const int32_t* eperm,
                       const int32_t* colptr, const int32_t* row, const int32_t* cpos, int64_t num_edges,
                       float negative_slope, const float* mask_edges, const float* mask_self,
                       const float* m, const float* inv_l, float* d_h, void* d_h_hi, void* d_h_lo,
                       float* d_a_src, float* d_a_dst, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* Attention scalars from the layer INPUT x [N, dim] instead of the projection: a_src[n,h] = <x[n,:], u[h,:]>,
 * a_dst[n,h] = <x[n,:], u[heads+h,:]> with u [2*heads, dim] the fold W_h^T att_*[h] (made by the caller).  Backward:
 * d_x [N, dim] = d_a u (written), d_u [2*heads, dim] = d_a^T x (deterministic).  With this, the backward of the
 * scores no longer modifies d(lin(x)), so etpgt_gat_bwd_mean can write that gradient directly as the split-bf16
 * operands d_h_hi / d_h_lo of the projection-gradient GEMMs (pass d_h = NULL). */
size_t etpgt_gat_input_scores_workspace_bytes(int64_t num_nodes, int dim, int heads);
int etpgt_gat_input_scores_fwd(const float* x, const float* u, int64_t num_nodes, int dim, int heads,
                               float* a_src, float* a_dst, etpgt_stream_t stream);
int etpgt_gat_input_scores_bwd(const float* x, const float* u, const float* d_a_src, const float* d_a_dst,
                               int64_t num_nodes, int dim, int heads, float* d_x, float* d_u,
                               void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* The node-wise parts of GATConv around the edge kernels, each one streaming pass (in PyTorch a dozen
 * element-wise / reduction launches over [N, heads*channels]):
 *   scores:    a_src[n,h] = <h[n,h,:], att_src[h,:]>, a_dst likewise (att_* are [heads*channels]);
 *   scores bwd: d_h (in/out) += d_a_src (x) att_src + d_a_dst (x) att_dst; d_att_src / d_att_dst [heads*channels]
 *              overwritten (deterministic column sums);
 *   head mean: out[n,:] = mean_h agg[n,h,:] + bias (bias [channels] or NULL) — concat=False, gat.py:92-107;
 *   head mean bwd: d_agg[n,h,:] = d_out[n,:] / heads, d_bias = column sums of d_out (or NULL).
 * One workspace size serves both backward calls. */
size_t etpgt_gat_aux_workspace_bytes(int64_t num_nodes, int width);
int etpgt_gat_scores_fwd(const float* h, const float* att_src, const float* att_dst, int64_t num_nodes,
                         int width, int heads, float* a_src, float* a_dst, etpgt_stream_t stream);
int etpgt_gat_scores_bwd(const float* h, const float* att_src, const float* att_dst, const float* d_a_src,
                         const float* d_a_dst, int64_t num_nodes, int width, int heads, float* d_h,
                         float* d_att_src, float* d_att_dst, void* ws, size_t ws_bytes, etpgt_stream_t stream);
int etpgt_head_mean_fwd(const float* agg, const float* bias, int64_t num_nodes, int heads, int channels,
                        float* out, etpgt_stream_t stream);
int etpgt_head_mean_bwd(const float* d_out, int64_t num_nodes, int heads, int channels, float* d_agg,
                        float* d_bias, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* PyG SAGEConv(aggr="mean") neighbour mean (etpgt/model/graphsage.py:43-48,75): mean_i = average of
 * x_j over in-edges (0 when there are none); backward distributes d_mean_i / indeg(i) to sources. */
int etpgt_sage_mean_fwd(const float* x, int64_t num_nodes, int dim, const int32_t* rowptr,
                        const int32_t* col, float* mean, etpgt_stream_t stream);
/* The same writing the mean directly as split-bf16 operands (mean = hi + lo) into rows of pitch `ld` elements — a
 * column block of the fused SAGEConv layer's [mean | x] GEMM operand; `mean` (fp32) may then be NULL. */
int etpgt_sage_mean_fwd_split(const float* x, int64_t num_nodes, int dim, const int32_t* rowptr,
                              const int32_t* col, float* mean, void* mean_hi, void* mean_lo, int64_t ld,
                              etpgt_stream_t stream);
int etpgt_sage_mean_bwd(const float* d_mean, int64_t num_nodes, int dim, const int32_t* rowptr,
                        const int32_t* colptr, const int32_t* row, float* d_x, etpgt_stream_t stream);
/* The same with the gradient of the mean given as the LEFT column half of a [N, ld] tensor and, optionally, the
 * root branch's gradient d_root (lin_r of SAGEConv; same pitch) added in: d_x = scatter(d_mean) + d_root.  This is
 * what the fused SAGEConv layer needs: one GEMM over [mean | x] produces both gradients side by side. */
int etpgt_sage_mean_bwd_ld(const float* d_mean, int64_t ld, const float* d_root, int64_t num_nodes, int dim,
                           const int32_t* rowptr, const int32_t* colptr, const int32_t* row, float* d_x,
                           etpgt_stream_t stream);

/* ---- a6: BatchNorm1d over node rows (+ residual, + ReLU) --------------------------------
 * graph_transformer.py:175-176, gat.py:138-140, graphsage.py:76-77.
 * stats: per-feature sums over this rank's rows, double precision: sums[0:dim] = sum x,
 * sums[dim:2dim] = sum x^2.  Under data parallelism the caller all-reduces `sums` (and the
 * row count) between stats and finalize so that the whole-batch semantics are kept. */
size_t etpgt_bn_workspace_bytes(int64_t n, int dim);
int etpgt_bn_stats(const float* x, int64_t n, int dim, double* sums,
                   void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* mean/invstd [dim] from sums and the GLOBAL row count; running stats updated in place
 * (momentum, unbiased variance) when running_mean != NULL. */
int etpgt_bn_finalize(const double* sums, double count, int dim, float eps, float momentum,
                      float* mean, float* invstd, float* running_mean, float* running_var,
                      etpgt_stream_t stream);
/* eval mode helper: mean/invstd from the running statistics. */
int etpgt_bn_from_running(const float* running_mean, const float* running_var, int dim, float eps,
                          float* mean, float* invstd, etpgt_stream_t stream);
/* y = (x-mean)*invstd*gamma + bias (+ residual) (then ReLU when relu != 0). */
int etpgt_bn_apply(const float* x, int64_t n, int dim, const float* mean, const float* invstd,
                   const float* gamma, const float* bias, const float* residual, int relu,
                   float* y, etpgt_stream_t stream);
/* The same with the layer's dropout fused in (etpgt/model/graph_transformer.py:176-177
 * `x = self.dropout_layer(x)`): y = dropout_p(bn(x) + residual) with a counter-based Philox4x32-10
 * mask keyed by (drop_seed, element index) that the backward entry points regenerate, so no mask is
 * stored; drop_p == 0 disables it.  y_hi / y_lo (both or neither): y also written split as bf16
 * pairs (y = hi + lo), the operand format of the next layer's tensor-core projection. */
int etpgt_bn_apply_ex(const float* x, int64_t n, int dim, const float* mean, const float* invstd,
                      const float* gamma, const float* bias, const float* residual, int relu,
                      double drop_p, uint64_t drop_seed, float* y, void* y_hi, void* y_lo,
                      etpgt_stream_t stream);
/* out[i] = 0 with probability p, else 1/(1-p) (Philox4x32-10 keyed by (seed, i / 4)): the attention
 * dropout masks (`alpha_mask` of etpgt_tconv_fwd, `mask_edges` / `mask_self` of etpgt_gat_fwd) of all
 * layers of one forward pass in a single launch.  out must be 16-byte aligned. */
int etpgt_dropout_mask(uint64_t seed, double p, int64_t n, float* out, etpgt_stream_t stream);
/* backward step 1: sums[0:dim] = sum g, sums[dim:2dim] = sum g*xhat with g = d_y (masked by
 * y > 0 when relu).  All-reduced across ranks by the caller in training mode. */
int etpgt_bn_bwd_stats(const float* x, const float* y, const float* d_y, int64_t n, int dim,
                       const float* mean, const float* invstd, int relu, double* sums,
                       void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* backward step 2: d_x; d_gamma/d_bias [dim] = LOCAL sums (pass the un-reduced sums as
 * local_sums).  training != 0 uses the batch-statistics formula with the GLOBAL count. */
int etpgt_bn_bwd_apply(const float* x, const float* y, const float* d_y, int64_t n, int dim,
                       const float* mean, const float* invstd, const float* gamma, int relu,
                       int training, const double* sums, double count, const double* local_sums,
                       float* d_x, float* d_gamma, float* d_bias, etpgt_stream_t stream);

/* Backward of etpgt_bn_apply_ex: g = d_y * dropout mask (* [y > 0] with relu); d_res (optional)
 * receives g, the gradient of the residual branch. */
int etpgt_bn_bwd_stats_ex(const float* x, const float* y, const float* d_y, int64_t n, int dim,
                          const float* mean, const float* invstd, int relu, double drop_p,
                          uint64_t drop_seed, double* sums, void* ws, size_t ws_bytes,
                          etpgt_stream_t stream);
int etpgt_bn_bwd_apply_ex(const float* x, const float* y, const float* d_y, int64_t n, int dim,
                          const float* mean, const float* invstd, const float* gamma, int relu,
                          int training, const double* sums, double count, const double* local_sums,
                          double drop_p, uint64_t drop_seed, float* d_x, float* d_res,
                          float* d_gamma, float* d_bias, etpgt_stream_t stream);

/* ---- a7: session readout (segmented reduction) ------------------------------------------
 * etpgt/model/base.py:136-193.  mode: 0 mean, 1 max, 2 last, 3 attention (softmax of the
 * caller-computed per-node `scores` inside each session).  Sessions are the contiguous node
 * ranges ptr[s]..ptr[s+1].  aux: argmax [S,dim] int32 for max, weights [N] float for attention. */
#define ETPGT_READOUT_MEAN 0
#define ETPGT_READOUT_MAX 1
#define ETPGT_READOUT_LAST 2
#define ETPGT_READOUT_ATTENTION 3
int etpgt_readout_fwd(const float* x, const int32_t* ptr, int64_t num_sessions, int dim, int mode,
                      const float* scores, float* out, void* aux, etpgt_stream_t stream);
int etpgt_readout_bwd(const float* x, const float* out, const float* d_out, const int32_t* ptr,
                      int64_t num_nodes, int64_t num_sessions, int dim, int mode, const void* aux,
                      float* d_x, float* d_scores, etpgt_stream_t stream);

/* ---- a8: sampled BPR / listwise / dual loss ---------------------------------------------
 * etpgt/train/losses.py:20-164, etpgt/model/base.py:80-113.
 * losses[3] = (alpha*listwise + (1-alpha)*bpr, listwise, bpr); mode 0 bpr (alpha ignored,
 * total = bpr), 1 listwise (total = listwise), 2 dual.  The means divide by total_sessions
 * (the GLOBAL batch under data parallelism).  scores [B, 1+num_neg] is saved for backward. */
#define ETPGT_LOSS_BPR 0
#define ETPGT_LOSS_LISTWISE 1
#define ETPGT_LOSS_DUAL 2
size_t etpgt_sampled_loss_workspace_bytes(int64_t batch, int num_neg, int dim);
int etpgt_sampled_loss_fwd(const float* sess, const float* table, const int64_t* targets,
                           const int64_t* negatives, int64_t batch, int num_neg, int dim,
                           int mode, float alpha, float temperature, double total_sessions,
                           float* scores, float* losses, void* ws, size_t ws_bytes,
                           etpgt_stream_t stream);
/* d_loss: device scalar (upstream gradient of losses[0]).  d_sess [B,dim] overwritten;
 * d_table dense [num_items,dim], caller-zeroed, rows ADDED deterministically. */
int etpgt_sampled_loss_bwd(const float* sess, const float* table, const int64_t* targets,
                           const int64_t* negatives, int64_t batch, int num_neg, int dim,
                           int mode, float alpha, float temperature, double total_sessions,
                           const float* scores, const float* d_loss, int64_t num_items,
                           int64_t padding_idx, float* d_sess, float* d_table, void* ws, size_t ws_bytes,
                           etpgt_stream_t stream);

/* ---- a8: full-catalogue softmax cross-entropy (tensor cores) ----------------------------
 * Replaces the listwise loss of etpgt/train/losses.py and the scoring of etpgt/model/base.py:80-113 with the
 * objective over the whole catalogue: z = sess . table^T / temperature over every item except padding_idx (-1: none),
 * lse[b] = logsumexp_j z[b, j], loss = sum_b (lse[b] - z[b, targets[b]]) / total_sessions (<= 0: batch; the GLOBAL
 * batch under data parallelism).  tcgen05 split-bf16 GEMMs with the softmax in the epilogue: the [batch, num_items]
 * logits are never materialised.  dim in {64, 128, 192, 256}; any batch >= 1, num_items >= 2.  Deterministic.
 * fwd: lse [batch] (saved for backward) and loss [1] are written.
 * bwd: d_loss is a device scalar.  d_sess [batch, dim] is overwritten; d_table_accumulate [num_items, dim] has
 * the table gradient ADDED (row padding_idx untouched).  Either may be NULL to skip it.  Both calls take the same
 * workspace size. */
size_t etpgt_full_softmax_workspace_bytes(int64_t batch, int64_t num_items, int dim);
int etpgt_full_softmax_fwd(const float* sess, const float* table, const int64_t* targets, int64_t batch,
                           int64_t num_items, int dim, float temperature, double total_sessions,
                           int64_t padding_idx, float* lse, float* loss, void* ws, size_t ws_bytes,
                           etpgt_stream_t stream);
int etpgt_full_softmax_bwd(const float* sess, const float* table, const int64_t* targets, const float* lse,
                           const float* d_loss, int64_t batch, int64_t num_items, int dim, float temperature,
                           double total_sessions, int64_t padding_idx, float* d_sess,
                           float* d_table_accumulate, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* Sampled softmax over ONE pool of num_sampled negatives shared by the batch, with the log-Q correction, on the same
 * tensor-core kernels.  pool_ids [M] ascending, inside [0, num_items); log_q [M] = log(M q(pool_ids[j])):
 *   z_pos[b] = sess_b . table[targets[b]] / T (fp32 gather-dot, no correction)
 *   z[b, j]  = sess_b . table[pool_ids[j]] / T - log_q[j], -inf where pool_ids[j] == targets[b] or == padding_idx
 *   lse[b]   = logsumexp(z_pos[b], z[b, :]),  loss = sum_b (lse[b] - z_pos[b]) / total_sessions (<= 0: batch)
 * dim in {64, 128, 192, 256}.  fwd writes lse, z_pos [batch] (both saved for backward) and loss [1].  bwd: d_loss is
 * a device scalar; d_sess [batch, dim] is overwritten and d_table_accumulate [num_items, dim] has the gradient of the
 * pool rows and target rows ADDED (row padding_idx untouched); either may be NULL.  Deterministic, no atomics, no
 * allocation, no synchronisation; both calls take the same workspace size. */
size_t etpgt_pool_softmax_workspace_bytes(int64_t batch, int64_t num_sampled, int dim);
int etpgt_pool_softmax_fwd(const float* sess, const float* table, const int64_t* targets, const int64_t* pool_ids,
                           const float* log_q, int64_t batch, int64_t num_items, int64_t num_sampled, int dim,
                           float temperature, double total_sessions, int64_t padding_idx, float* lse, float* z_pos,
                           float* loss, void* ws, size_t ws_bytes, etpgt_stream_t stream);
int etpgt_pool_softmax_bwd(const float* sess, const float* table, const int64_t* targets, const int64_t* pool_ids,
                           const float* log_q, const float* lse, const float* z_pos, const float* d_loss,
                           int64_t batch, int64_t num_items, int64_t num_sampled, int dim, float temperature,
                           double total_sessions, int64_t padding_idx, float* d_sess, float* d_table_accumulate,
                           void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* Precision of both softmax losses.  The four calls above are the _ex calls with ETPGT_SOFTMAX_BF16X3.
 * ETPGT_SOFTMAX_BF16X3: every product is split-bf16 (x = hi + lo, hi.hi + hi.lo + lo.hi, fp32 accumulation), ~1e-5
 *   relative to the fp64 objective.
 * ETPGT_SOFTMAX_BF16: a different numerical contract, for training.  S (sess), E (the table rows, or the gathered pool
 *   rows) and G = (P - onehot) / (T B_total) are each rounded once to bf16 (round to nearest even) and every product
 *   is one bf16 MMA with fp32 accumulation.  Everything else is as above: lse, the online max and sum and the target
 *   logit in fp32; the pool's log_q, padding entries and hits; the pool's positive is the fp32 gather-dot of the
 *   rounded operands, z_pos = bf16(s_b) . bf16(e_t) / T, with gradient terms c_b bf16(e_t) into d_sess and
 *   c_b bf16(s_b) into the table, where c_b = (exp(z_pos - lse) - 1) d_loss / (T B_total) is the positive's entry of G
 *   and rounded to bf16 like the rest of G (products of two bf16 values are exact in fp32), so a pool of every
 *   non-padding item with log_q = 0 is still the bf16 full loss.  Deterministic, no atomics.  lse and the loss are
 *   within ~1e-4 of the fp64 objective of the rounded S and E.
 * The _ex calls take the workspace of etpgt_full_softmax_workspace_bytes / etpgt_pool_softmax_workspace_bytes in both
 * precisions: a bf16 call needs no more (it uses less).  Any other precision returns ETPGT_EINVAL. */
#define ETPGT_SOFTMAX_BF16X3 0
#define ETPGT_SOFTMAX_BF16 1
int etpgt_full_softmax_fwd_ex(const float* sess, const float* table, const int64_t* targets, int64_t batch,
                              int64_t num_items, int dim, float temperature, double total_sessions,
                              int64_t padding_idx, float* lse, float* loss, void* ws, size_t ws_bytes,
                              etpgt_stream_t stream, int precision);
int etpgt_full_softmax_bwd_ex(const float* sess, const float* table, const int64_t* targets, const float* lse,
                              const float* d_loss, int64_t batch, int64_t num_items, int dim, float temperature,
                              double total_sessions, int64_t padding_idx, float* d_sess,
                              float* d_table_accumulate, void* ws, size_t ws_bytes, etpgt_stream_t stream,
                              int precision);
int etpgt_pool_softmax_fwd_ex(const float* sess, const float* table, const int64_t* targets, const int64_t* pool_ids,
                              const float* log_q, int64_t batch, int64_t num_items, int64_t num_sampled, int dim,
                              float temperature, double total_sessions, int64_t padding_idx, float* lse, float* z_pos,
                              float* loss, void* ws, size_t ws_bytes, etpgt_stream_t stream, int precision);
int etpgt_pool_softmax_bwd_ex(const float* sess, const float* table, const int64_t* targets, const int64_t* pool_ids,
                              const float* log_q, const float* lse, const float* z_pos, const float* d_loss,
                              int64_t batch, int64_t num_items, int64_t num_sampled, int dim, float temperature,
                              double total_sessions, int64_t padding_idx, float* d_sess, float* d_table_accumulate,
                              void* ws, size_t ws_bytes, etpgt_stream_t stream, int precision);

/* ---- a9/a10: full-catalogue scoring with fused top-k and metrics ------------------------
 * etpgt/model/base.py:59-78, etpgt/utils/metrics.py:6-66.  Scores are never materialised.
 * Ties go to the lower item id.  id_base offsets the ids of an item-table shard.
 * k bounds: the tensor-core scorer and both merges take 1 <= k <= ETPGT_SCORE_MAX_K; the fp32 CUDA-core scorer takes
 * 1 <= k <= 64.  A larger k returns ETPGT_EINVAL. */
#define ETPGT_SCORE_MAX_K 256
size_t etpgt_score_topk_workspace_bytes(int64_t batch, int64_t num_items, int dim, int k);
/* fp32 CUDA-core path (exact reference arithmetic, small batches). */
int etpgt_score_topk_f32(const float* sess, const float* table, int64_t batch, int64_t num_items,
                         int dim, int k, int64_t id_base, float* top_val, int64_t* top_idx,
                         void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* Tensor-core path: bf16 operands (row-major [rows, dim], 16-byte aligned, dim in {64,128,192,256}),
 * fp32 accumulation in TMEM, tcgen05.mma fed by TMA, top-k (k <= ETPGT_SCORE_MAX_K) fused into the TMEM epilogue.
 * The workspace grows with k: for k > 32 it holds a slot for every 16-item piece of the catalogue per session row
 * (72 bytes per 16 items), so callers score large batches in row chunks (etpgt_b200.ops.score_topk does).
 * Oracle: fp64 scores of the bf16-rounded operands (oracle/model_ref.predict(bf16_inputs=True)). */
int etpgt_f32_to_bf16(const float* src, void* dst_bf16, int64_t n, etpgt_stream_t stream);
size_t etpgt_score_topk_bf16_workspace_bytes(int64_t batch, int64_t num_items, int k);
int etpgt_score_topk_bf16(const void* sess_bf16, const void* table_bf16, int64_t batch, int64_t num_items,
                          int dim, int k, int64_t id_base, float* top_val, int64_t* top_idx,
                          void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* The same with the evaluation metric's input fused into the select epilogue (SURVEY.md K8): with targets [batch],
 * hit_pos[b] = position of targets[b] among the row's k results (first match, etpgt/utils/metrics.py:49) or -1,
 * taken from the registers that hold the sorted list — the [batch, k] id matrix is not read again.
 * etpgt_hit_metrics turns hit_pos into the Recall@k / NDCG@k counters for any k <= the k scored. */
int etpgt_score_topk_bf16_eval(const void* sess_bf16, const void* table_bf16, int64_t batch, int64_t num_items,
                               int dim, int k, int64_t id_base, float* top_val, int64_t* top_idx,
                               const int64_t* targets, int32_t* hit_pos, void* ws, size_t ws_bytes,
                               etpgt_stream_t stream);
/* Filtered scoring: the same results with each row's listed ids left out (a session's own items, the padding id).
 * exclude: int64 [batch, exclude_width], row-major, one row per session; each row sorted ascending, duplicates
 * allowed, ids outside [id_base, id_base + num_items) ignored (so an item shard takes the global list unchanged and
 * rows may be padded with -1).  exclude_width == 0 excludes nothing.  Unlike the unfiltered entry points k may exceed
 * the eligible items of a row: the missing slots are (-inf, INT64_MAX).  An excluded target gets hit_pos -1.
 * bf16: same workspace as etpgt_score_topk_bf16_workspace_bytes, exclude_width <= 16384; targets / hit_pos
 * nullable. */
int etpgt_score_topk_bf16_exclude(const void* sess_bf16, const void* table_bf16, int64_t batch, int64_t num_items,
                                  int dim, int k, int64_t id_base, float* top_val, int64_t* top_idx,
                                  const int64_t* targets, int32_t* hit_pos, const int64_t* exclude,
                                  int64_t exclude_width, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* fp32: same workspace as etpgt_score_topk_workspace_bytes. */
int etpgt_score_topk_f32_exclude(const float* sess, const float* table, int64_t batch, int64_t num_items, int dim,
                                 int k, int64_t id_base, float* top_val, int64_t* top_idx, const int64_t* exclude,
                                 int64_t exclude_width, void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* exact merge of `parts` candidate lists per row ([B, parts*k] values + ids). */
int etpgt_topk_merge(const float* cand_val, const int64_t* cand_idx, int64_t batch, int parts, int k,
                     float* top_val, int64_t* top_idx, etpgt_stream_t stream);
/* hits/ndcg accumulators: out[0] += #hits@k, out[1] += sum 1/log2(pos+2) (double[2], caller-zeroed). */
int etpgt_topk_metrics(const int64_t* top_idx, const int64_t* targets, int64_t batch, int k_stride,
                       int k, double* out, etpgt_stream_t stream);
/* Item-sharded evaluation (SURVEY.md §8e): every rank scores ALL sessions against its contiguous id range and
 * packs its candidates as one block (val [rows_total, k] f32 at offset 0, idx [rows_total, k] i64 at idx_offset);
 * ONE all-gather lays the blocks out rank-major (part p at parts + p * part_stride).  This merges rows
 * [row_begin, row_begin + rows) out of that layout exactly (score desc, id asc).  With targets [rows] it also
 * writes hit_pos[r] = position of targets[r] in the merged top-k or -1 — the input of etpgt_hit_metrics, which
 * adds (#hits within k, sum of 1/log2(pos+2)) to out[0], out[1] (etpgt/utils/metrics.py:6-66) without the
 * [rows, k] id matrix being read again. */
int etpgt_topk_merge_parts(const void* parts, int num_parts, size_t part_stride, size_t idx_offset,
                           int64_t rows_total, int k, int64_t row_begin, int64_t rows, float* top_val,
                           int64_t* top_idx, const int64_t* targets, int32_t* hit_pos, etpgt_stream_t stream);
int etpgt_hit_metrics(const int32_t* hit_pos, int64_t batch, int k, double* out, etpgt_stream_t stream);

/* ---- generic helper shared by embedding / loss backward ---------------------------------
 * d_table[key] += sum_{p: keys[p]==key} coef[p] * src[p / src_div]  in ascending p, one writer
 * per row (deterministic).  coef may be NULL (=1); row skip_key (-1 = none) is left untouched.  dim in
 * {32, 64, 128, 192, 256}. */
size_t etpgt_scatter_rows_workspace_bytes(int64_t m);
int etpgt_scatter_rows(const int64_t* keys, const float* coef, const float* src, int64_t m,
                       int src_div, int dim, int64_t num_rows, int64_t skip_key, float* d_table,
                       void* ws, size_t ws_bytes, etpgt_stream_t stream);

/* ---- a11 / §8(f1): the optimizer step ------------------------------------------------------
 * torch.optim.AdamW (scripts/train/train_baseline.py:252-256, stepped at etpgt/train/trainer.py:127)
 * and torch.optim.Adam (scripts/pipeline/run_full_pipeline.py:210) over a list of fp32 tensors in ONE
 * launch (chunks of <= 48 tensors).  `tensors` is a HOST array, read during the call.  decoupled != 0:
 * AdamW (p *= 1 - lr*wd); 0: Adam with L2 (g += wd*p).  `step` is the 1-based step count shared by
 * the listed tensors (bias corrections are computed from it in double, as torch does on the host).
 * zero_grad != 0 also clears every listed gradient (persistent gradient buffers that the next
 * backward accumulates into).  Dense semantics: every element of every tensor is updated. */
typedef struct etpgt_adam_tensor {
  float* param;
  float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int64_t numel;
} etpgt_adam_tensor;
int etpgt_adam_step(const etpgt_adam_tensor* tensors, int count, double lr, double beta1, double beta2,
                    double eps, double weight_decay, int decoupled, int64_t step, int zero_grad,
                    etpgt_stream_t stream);
/* Row-sparse ("lazy") AdamW / Adam over ONE [rows, dim] fp32 table with a dense gradient buffer.  A row is
 * touched iff an element of its gradient row compares != 0 (+0 / -0 do not, NaN does).  Every element of a
 * touched row gets exactly the etpgt_adam_step update (decoupled / L2 decay of touched rows only, bias
 * corrections from the global `step`) and, with zero_grad != 0, its gradient row is cleared; an untouched
 * row's parameter and moments are neither read nor written.  NOT equivalent to the dense step (which decays
 * and moves every row).  Bytes: rows*dim*4 + touched*dim*28.  dim in {32, 64, 128, 256} needs 16-byte aligned
 * buffers; any other dim >= 1 takes a scalar path.  `touched` (optional, device int64) receives the number of
 * rows updated.  No allocation, no synchronisation. */
int etpgt_adam_rows(float* param, float* grad, float* exp_avg, float* exp_avg_sq, int64_t rows, int dim,
                    double lr, double beta1, double beta2, double eps, double weight_decay, int decoupled,
                    int64_t step, int zero_grad, int64_t* touched, etpgt_stream_t stream);
/* torch.optim.SparseAdam's arithmetic (torch/optim/_functional.py::sparse_adam, one fp32 rounding per torch
 * op, no contraction; step_size = lr*sqrt(1-b2^step)/(1-b1^step) formed in double; maximize negates g) over
 * one [rows, dim] table.  Two modes:
 *   indices == NULL (scan): `grad` is a dense [rows, dim] buffer; touched rows as etpgt_adam_rows, cleared
 *     with zero_grad != 0.
 *   indices != NULL (listed): a coalesced sparse gradient, `indices` [nnz] strictly ascending rows and `grad`
 *     its values [nnz, dim]; every listed row is updated (all-zero ones too: torch's index-set semantics),
 *     listed rows outside [0, rows) are skipped; zero_grad must be 0.
 * Alignment, `touched`, allocation and synchronisation as etpgt_adam_rows. */
int etpgt_sparse_adam(float* param, float* exp_avg, float* exp_avg_sq, int64_t rows, int dim, float* grad,
                      const int64_t* indices, int64_t nnz, double lr, double beta1, double beta2, double eps,
                      int maximize, int64_t step, int zero_grad, int64_t* touched, etpgt_stream_t stream);

/* ---- §8(f3): co-occurrence graph construction ----------------------------------------------
 * scripts/data/04_build_graph.py:25-127 (`build_co_event_graph`): sessions are
 * sess_items[sess_ptr[s] : sess_ptr[s+1]] in timestamp order (the reference's groupby + sort); every
 * pair of events at most `window` steps apart adds one co-occurrence to the undirected edge
 * (min item, max item); count = co-occurrences, last_ts = max(0, timestamps of the event holding the
 * smaller item id) (timestamps / last_ts may both be NULL).  Edges come out ordered by count
 * descending, ties by first emission (the stable order of the reference's dict; pandas' default sort
 * leaves ties unspecified).  Outputs hold `capacity` entries; *num_edges (device scalar) receives the
 * true edge count (<= num_events * window) and at most `capacity` edges are written.  The per-edge
 * `event_pair_hist` of the reference is not produced (unused by the training path). */
size_t etpgt_cooc_graph_workspace_bytes(int64_t num_events, int window);
int etpgt_cooc_graph_build(const int64_t* sess_ptr, const int64_t* sess_items, const int64_t* timestamps,
                           int64_t num_sessions, int64_t num_events, int window, int64_t num_items,
                           int64_t capacity, int64_t* item_i, int64_t* item_j, int64_t* count,
                           int64_t* last_ts, int64_t* num_edges, void* ws, size_t ws_bytes,
                           etpgt_stream_t stream);

/* Scatter plans: the sort of a scatter depends on its keys only, and the keys of both scatters of a
 * training step (the batch's node ids for the embedding backward; [target | negatives] per session for the
 * loss backward) are fixed once the batch exists.  etpgt_scatter_plan sorts them once per batch (next to
 * the CSR / CSC index, off the step's critical path): sorted_key [m], perm [m] (stable).  The *_planned
 * entry points then only run the owner-per-row accumulation.  Loss keys are laid out
 * [b][0] = target, [b][1 + c] = negative c. */
size_t etpgt_scatter_plan_workspace_bytes(int64_t m);
int etpgt_scatter_plan(const int64_t* keys, int64_t m, int64_t num_rows, int32_t* sorted_key, int32_t* perm,
                       void* ws, size_t ws_bytes, etpgt_stream_t stream);
/* the plan of the loss scatter straight from targets [B] and negatives [B, num_neg] (m = B * (1 + num_neg)) */
int etpgt_scatter_plan_loss(const int64_t* targets, const int64_t* negatives, int64_t batch, int num_neg,
                            int64_t num_rows, int32_t* sorted_key, int32_t* perm, void* ws, size_t ws_bytes,
                            etpgt_stream_t stream);
int etpgt_scatter_rows_planned(const int32_t* sorted_key, const int32_t* perm, const float* coef,
                               const float* src, int64_t m, int src_div, int dim, int64_t skip_key,
                               float* d_table, etpgt_stream_t stream);
/* Item ids index the table and its gradient buffer raw (the reference's nn.Embedding raises IndexError for
 * an id >= num_items, etpgt/model/base.py:36).  *flag |= 1 (device int32, caller-zeroed, sticky) when any id of
 * up to three lists (node ids, targets, negatives; NULL / 0 to skip) lies outside [0, num_rows).  Asynchronous:
 * the host reads the flag when it wants to (ops.prepare_batch runs the check per batch on the preparation stream,
 * the trainer reads the flag once per epoch). */
int etpgt_ids_check(const int64_t* a, int64_t na, const int64_t* b, int64_t nb, const int64_t* c, int64_t nc,
                    int64_t num_rows, int32_t* flag, etpgt_stream_t stream);
/* Batch preparation in one call: etpgt_csr_from_coo of (src, dst) plus the scatter plans of `ids` [N] (rows of
 * num_items) and of the loss keys ([b][0] = targets[b], [b][1 + c] = negatives[b][c]; targets == NULL skips that
 * plan), with identical outputs — but the destination sort and the two plan sorts run as ONE segmented radix sort
 * (the segment number rides above the key bits), so the call costs two sorts instead of four. */
size_t etpgt_batch_prepare_workspace_bytes(int64_t num_edges, int64_t num_nodes, int64_t num_loss_keys);
int etpgt_batch_prepare(const int64_t* src, const int64_t* dst, int64_t num_edges, int64_t num_nodes,
                        const int64_t* ids, const int64_t* targets, const int64_t* negatives,
                        int64_t num_sessions, int num_neg, int64_t num_items, int32_t* rowptr, int32_t* col,
                        int32_t* eperm, int32_t* colptr, int32_t* row, int32_t* cpos, int32_t* nodes_key,
                        int32_t* nodes_perm, int32_t* loss_key, int32_t* loss_perm, void* ws, size_t ws_bytes,
                        etpgt_stream_t stream);
int etpgt_embed_pe_bwd_planned(const int64_t* ids, int64_t n, const float* d_out, int64_t num_items,
                               const float* pe, int pe_per_node, int k_pe, int dim, int64_t padding_idx,
                               const int32_t* plan_sorted_key, const int32_t* plan_perm, float* d_table,
                               float* d_w_pe, float* d_b_pe, void* ws, size_t ws_bytes, etpgt_stream_t stream);
int etpgt_sampled_loss_bwd_planned(const float* sess, const float* table, const int64_t* targets,
                                   const int64_t* negatives, int64_t batch, int num_neg, int dim,
                                   int mode, float alpha, float temperature, double total_sessions,
                                   const float* scores, const float* d_loss, int64_t num_items,
                                   int64_t padding_idx, const int32_t* plan_sorted_key,
                                   const int32_t* plan_perm, float* d_sess, float* d_table, void* ws,
                                   size_t ws_bytes, etpgt_stream_t stream);

/* ---- (e) multi-GPU: peer-memory communicator ----------------------------------------------------
 * Session-batch data parallelism over one NVSwitch box (SURVEY.md §8e; the reference trains on one GPU,
 * etpgt/train/trainer.py:69-131).  One process per GPU; every rank owns one device *region* (cudaMalloc,
 * zeroed control block of etpgt_comm_control_bytes() at its start, the rest is the caller's: gradient and
 * parameter buffers that peers read / write) and maps the regions of all peers — over CUDA IPC
 * (etpgt_comm_ipc_handle on every rank, handles exchanged by the host, etpgt_comm_connect_ipc), or by plain
 * pointers when several ranks live in one process (etpgt_comm_connect_ptrs).  The kernels below move data
 * with ordinary loads / stores over NVLink and order it with system-scope flags; every cross-rank sum runs in
 * rank order on every rank, so replicas stay bit-identical.  All ranks must issue the same sequence of
 * communicator calls (per barrier channel; the small all-reduce has one sequence), each sequence on ONE
 * stream.  A wait that sees no peer for the time-out (default 30 s) gives
 * up and records it in the status word (etpgt_comm_status) instead of hanging the GPU; later waits of that rank
 * return at once.
 *   barrier        everything this rank issued before (on that stream) is complete and visible to its peers, and
 *                  vice versa; `channel` 0..3 selects an independent barrier sequence, one per stream that
 *                  synchronises (all ranks use the same channel for the same purpose)
 *   allreduce_f64  out[i] = sum_r in_r[i], count <= 520 doubles (BatchNorm statistics), ONE single-CTA kernel
 *                  (in == out allowed)
 *   sum_f32        out[i] = sum_r region_r[offset + 4*i]: the dense-gradient exchange (callers bracket it
 *                  with barriers: sources complete before, sources reusable after) */
#define ETPGT_MAX_RANKS 8
#define ETPGT_IPC_HANDLE_BYTES 64
typedef struct etpgt_comm etpgt_comm_t;
size_t etpgt_comm_control_bytes(void);
int etpgt_comm_create(int rank, int world, size_t region_bytes, etpgt_comm_t** out);
int etpgt_comm_ipc_handle(const etpgt_comm_t* comm, unsigned char* handle /* [ETPGT_IPC_HANDLE_BYTES] */);
int etpgt_comm_connect_ipc(etpgt_comm_t* comm, const unsigned char* handles /* [world][ETPGT_IPC_HANDLE_BYTES] */);
int etpgt_comm_connect_ptrs(etpgt_comm_t* comm, void* const* bases /* [world] */);
void* etpgt_comm_region(const etpgt_comm_t* comm, int rank);
int etpgt_comm_set_timeout(etpgt_comm_t* comm, double seconds);
int etpgt_comm_destroy(etpgt_comm_t* comm);
int etpgt_comm_barrier(const etpgt_comm_t* comm, int channel, etpgt_stream_t stream);
int etpgt_comm_allreduce_f64(const etpgt_comm_t* comm, const double* in, double* out, int count,
                             etpgt_stream_t stream);
int etpgt_comm_sum_f32(const etpgt_comm_t* comm, size_t offset, int64_t numel, float* out, etpgt_stream_t stream);
int etpgt_comm_status(const etpgt_comm_t* comm, int* status);
/* The item table under data parallelism: reduce-scatter of its gradient + dense AdamW / Adam + all-gather of
 * the updated rows as ONE kernel over peer memory (replaces an 84 MB / 1 GB NCCL all-reduce followed by a
 * replicated optimizer pass; reference semantics: dense decoupled decay over every row,
 * scripts/train/train_baseline.py:252-256).  The table [rows, dim] lives at param_offset and its gradient at
 * grad_offset of EVERY rank's region.  This rank owns rows [row_begin, row_end): it sums those rows of all
 * ranks' gradients (rank order), updates them with its moments exp_avg / exp_avg_sq ([rows, dim], only the
 * owned rows are read and written) and stores the new values into every rank's table.  Arithmetic and
 * hyper-parameters as etpgt_adam_step.  Bracket with etpgt_comm_barrier: gradients complete before; all
 * tables complete and all gradient buffers free to be cleared after. */
int etpgt_dp_adam_table(const etpgt_comm_t* comm, size_t param_offset, size_t grad_offset, float* exp_avg,
                        float* exp_avg_sq, int64_t rows, int dim, int64_t row_begin, int64_t row_end, double lr,
                        double beta1, double beta2, double eps, double weight_decay, int decoupled, int64_t step,
                        etpgt_stream_t stream);

/* ---- a11: step driver --------------------------------------------------------------------------
 * One host call for the whole training step of graph_transformer_optimized — what Trainer.train_epoch
 * (etpgt/train/trainer.py:95-127) runs between `optimizer.zero_grad()` and `optimizer.step()`:
 * model(batch) (etpgt/model/graph_transformer.py:126-182, use_ffn=False), the sampled loss
 * (etpgt/train/losses.py) and the backward pass.  It launches exactly the entry points above, in the order and
 * with the arguments of the per-operator path, out of one caller-provided arena; results are bit-identical to
 * calling them one by one.
 *
 * All pointers are device pointers except the descriptor itself (host).  Gradient outputs are OVERWRITTEN,
 * except d_table whose rows are ADDED (caller-zeroed, or the optimizer's persistent gradient buffer).
 * layer[l].weight / bias are the query|key|value|skip blocks as one [4*dim, dim] / [4*dim] buffer.
 * Dropout: attention-weight masks from (alpha_seed, alpha_p), layer dropout from (drop_seed, drop_p), both
 * Philox4x32-10 as in etpgt_dropout_mask / etpgt_bn_apply_ex; ignored when training == 0.
 * plan_* (optional): etpgt_scatter_plan of `ids` and of the [target | negatives] keys.
 *
 * Phases (data parallelism): the step is cut at the BatchNorm statistics exchanges, and once more after the last
 * kernel that adds to d_table, into 2*layers+2 phases; run [phase_begin, phase_end) per call.  bn_sums is
 * [2*layers][2*dim+1] doubles: row l = forward sums of layer l (produced by phase l), row layers+l = backward
 * sums of layer l (produced by phase 2*layers-1-l).  With distributed != 0 the caller all-reduces the row a
 * phase produced before running the next phase (the row's last element carries the row count); d_table is
 * complete after phase 2*layers, so its all-reduce can overlap phase 2*layers+1 (weight gradient of layer 0 and
 * the PE projection gradient).  With distributed == 0 run all phases in one call.
 * With distributed != 0 AND comm != NULL the driver exchanges the rows itself (etpgt_comm_allreduce_f64 between
 * the statistics kernel and the apply kernel): no cuts are needed, run all phases in one call. */
#define ETPGT_GT_MAX_LAYERS 4
typedef struct etpgt_gt_layer {
  const float* weight;       /* [4*dim, dim] */
  const float* bias;         /* [4*dim] */
  const float* w_beta;       /* [3*dim] or NULL (beta=False) */
  const float* bn_weight;    /* [dim] */
  const float* bn_bias;      /* [dim] */
  float* running_mean;       /* [dim], updated in training */
  float* running_var;        /* [dim] */
  int64_t* num_batches_tracked; /* scalar, +1 in training (may be NULL) */
  float* d_weight;           /* [4*dim, dim] */
  float* d_bias;             /* [4*dim] */
  float* d_w_beta;           /* [3*dim] or NULL */
  float* d_bn_weight;        /* [dim] */
  float* d_bn_bias;          /* [dim] */
  double momentum, eps;
  uint64_t alpha_seed, drop_seed;
} etpgt_gt_layer_t;

typedef struct etpgt_gt_step {
  int64_t struct_bytes;      /* sizeof(etpgt_gt_step_t): guards against header / binding drift */
  /* batch (PyG collate layout) and its index (etpgt_csr_from_coo) */
  int64_t num_nodes, num_edges, num_sessions;
  const int64_t* ids;        /* [N] item id per node */
  const int64_t* batch_vec;  /* [N] session index per node, non-decreasing */
  const int32_t *rowptr, *col, *eperm, *colptr, *row, *cpos;
  const int64_t* targets;    /* [B] */
  const int64_t* negatives;  /* [B, num_neg] */
  const int32_t *plan_nodes_key, *plan_nodes_perm, *plan_loss_key, *plan_loss_perm; /* or NULL */
  /* model */
  int64_t num_items, padding_idx;
  int32_t dim, heads, num_layers, k_pe, num_neg, readout_mode, loss_mode;
  int32_t training, backward, distributed;
  float alpha, temperature;
  double total_sessions, alpha_p, drop_p;
  const float* table;        /* [num_items, dim] */
  const float* pe;           /* [num_items, k_pe] cached Laplacian PE or NULL */
  const float* w_pe;         /* [dim, k_pe] */
  const float* b_pe;         /* [dim] */
  float* d_table;            /* [num_items, dim] rows ADDED */
  float* d_w_pe;             /* [dim, k_pe] */
  float* d_b_pe;             /* [dim] */
  etpgt_gt_layer_t layer[ETPGT_GT_MAX_LAYERS];
  /* outputs / exchange */
  float* sess;               /* [B, dim] session embeddings */
  float* losses;             /* [3] (total, listwise, bpr) */
  double* bn_sums;           /* [2*layers][2*dim+1] */
  const etpgt_comm_t* comm;  /* peer-memory communicator for the BatchNorm exchange, or NULL */
  void* arena;
  size_t arena_bytes;        /* >= etpgt_gt_step_arena_bytes */
} etpgt_gt_step_t;

size_t etpgt_gt_step_arena_bytes(const etpgt_gt_step_t* step);
int etpgt_gt_step_num_phases(const etpgt_gt_step_t* step);
int etpgt_gt_step_run(const etpgt_gt_step_t* step, int phase_begin, int phase_end, etpgt_stream_t stream);

/* The same phases as ONE CUDA graph launch, for small batches (the reference trains at 32 sessions per step,
 * params.yaml:6) where the step is bound by the ~55 launch gaps between microsecond kernels: the driver's launches
 * are captured from `stream` (which must not be the legacy default stream), the capture updates the executable
 * graph kept in `cache` in place (kernel arguments / grids / variants change from batch to batch, the topology does
 * not; it is rebuilt when it does) and is launched once.  Bit-identical to etpgt_gt_step_run.  A cache belongs to
 * one model / stream; etpgt_graph_rebuilds counts instantiations (1 in a steady loop). */
typedef struct etpgt_graph etpgt_graph_t;
int etpgt_graph_create(etpgt_graph_t** out);
int etpgt_graph_destroy(etpgt_graph_t* cache);
int64_t etpgt_graph_rebuilds(const etpgt_graph_t* cache);
int etpgt_gt_step_run_graph(const etpgt_gt_step_t* step, int phase_begin, int phase_end, etpgt_graph_t* cache,
                            etpgt_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ETPGT_B200_H */
