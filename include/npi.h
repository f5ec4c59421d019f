/* libnpi -- C ABI of the B200-native NPI-GNN hot path (sm_100a).
 *
 * The reference (AshuiRUA/NPI-GNN) is pure Python and has no FFI of its own; the boundary
 * this library sits behind is the torch-geometric operator API that the reference's model
 * and trainers call (SURVEY.md section 8b).  Every entry point below names the reference
 * interface it replaces (paths relative to the reference root).  INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *  - every function returns int: 0 = NPI_OK, negative = NPI_ERR_*; text via npi_last_error()
 *    (thread-local).  No C++ exception crosses the boundary.
 *  - the CALLER allocates everything (inputs, outputs, workspaces); nothing is retained
 *    past the call.  Pointers are DEVICE pointers unless the name ends in _h (host).
 *  - every call takes the CUDA stream (cudaStream_t as void*) and is asynchronous; no call
 *    synchronises, allocates or frees, so a sequence of calls can be captured in a CUDA graph.
 *  - data-dependent sizes are read from device memory: a size argument comes as a pair
 *    (`const int32_t* n_dev`, `int32_t n_host`); if n_dev is non-NULL the kernel uses *n_dev
 *    and n_host is only an upper bound used for nothing but sanity checks.
 *  - indices are int32, features float32 row-major, hidden width is 128.
 *  - determinism: no floating-point atomics anywhere; identical inputs give bit-identical
 *    outputs on the same device.
 */
#ifndef NPI_H_
#define NPI_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NPI_OK 0
#define NPI_ERR_INVALID (-1)
#define NPI_ERR_CUDA (-2)
#define NPI_ERR_WORKSPACE (-3)

#define NPI_HIDDEN 128

typedef void* npi_stream_t;

const char* npi_last_error(void);
int npi_version(void);
/* number of SMs of the current device (148 on B200); host query, no stream work */
int npi_sm_count(int32_t* out_h);

/* ------------------------------------------------------------------------------------------
 * Node features of a batch, either dense or "virtual".
 * Replaces the x tensor the reference materialises per subgraph in
 * src/classes.py:706-717 + 728 (x[i] = [structural label | node2vec emb | k-mer]).
 *   dense  : x != NULL, row i at x + i*ldx, F columns.
 *   virtual: x == NULL; x[i][0] = (float)dist[i], x[i][c] = table[gid[i]*ld + c] for 1<=c<F.
 *            The table keeps column 0 free for the label, ld is a multiple of 4 and rows are
 *            16-byte aligned, columns >= F are zero.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    const float* x;
    int32_t ldx;
    const float* table;
    int32_t ld;
    const int32_t* gid;
    const uint8_t* dist;
    int32_t F;
} npi_features_t;

/* ------------------------------------------------------------------------------------------
 * Graph preparation (host, once per dataset).
 * Replaces the Node.interaction_list object graph built in src/generate_edgelist.py:56-90
 * and src/generate_dataset.py:204-216.  edges_h[2*i] = RNA serial, edges_h[2*i+1] = protein
 * serial, in the order the reference appends interactions.  Duplicate keys keep their first
 * position (the reference collects keys in a set, src/classes.py:667).  Outputs: CSR with
 * adjacency in that order, the undirected edge id of every CSR entry, and for each input
 * edge its de-duplicated id (or -1 for a repeated key).  All arrays are HOST memory;
 * rowptr_h[V+1], col_h/eid_h[2*E], edge_id_h[E].
 * ------------------------------------------------------------------------------------------ */
int npi_csr_build_host(const int32_t* edges_h, int64_t num_edges, int32_t num_nodes,
                       int32_t* rowptr_h, int32_t* col_h, int32_t* eid_h, int32_t* edge_id_h,
                       int64_t* num_unique_h);

/* ------------------------------------------------------------------------------------------
 * h-hop enclosing-subgraph extraction (GPU frontier BFS).
 * Replaces LncRNA_Protein_Interaction_dataset_1hop_1220_InMemory.local_subgraph_generation
 * (src/classes.py:652-733) generalised to h hops per SURVEY.md Appendix B.
 *   colm[k] = col[k] with bit 31 set  <=>  the edge of CSR entry k is in
 *             set_allInteractionKey_cannotUse (src/generate_dataset.py:297-299; tested at
 *             src/classes.py:681,690) -- produced by npi_csr_fold_mask from (col, eid, mask).
 *   pairs[2*i], pairs[2*i+1] = (RNA serial, protein serial) of target pair i.
 * Local node 0 = RNA, 1 = protein, then BFS discovery order; dist = hop distance = structural
 * label.  Subgraph adjacency is emitted as CSR by destination over local ids offset by the
 * batch position (row graph_ptr[i]+k), canonical row order: partner target first for the two
 * targets, then unmasked neighbours in adjacency order that share an edge of the subgraph.
 * The per-pair working set lives in shared memory when 4*(5V+1)+V bytes fit (V <~ 9.7 k nodes);
 * larger graphs use `workspace` (npi_khop_workspace_bytes, one slab per CTA).
 * ------------------------------------------------------------------------------------------ */
int npi_csr_fold_mask(const int32_t* col, const int32_t* eid, const uint8_t* mask, int64_t nnz,
                      int32_t* colm, npi_stream_t stream);
int64_t npi_khop_workspace_bytes(int32_t num_nodes, int32_t num_ctas);
/* pass 1: n_out[i] = nodes, e_out[i] = directed edges of subgraph i */
int npi_khop_count(const int32_t* rowptr, const int32_t* colm, int32_t num_nodes,
                   const int32_t* pairs, int32_t num_pairs, int32_t h,
                   int32_t* n_out, int32_t* e_out,
                   void* workspace, int64_t workspace_bytes, int32_t num_ctas, npi_stream_t stream);
/* pass 2: graph_ptr[P+1] / edge_ptr[P+1] are the exclusive scans of the pass-1 counts and
 * max_graph_nodes >= max_i n_out[i].  Writes gid[N], dist[N], sub_rowptr[N+1] (batch-global edge
 * offsets), sub_col[E] (batch-global node ids).  n_capacity / e_capacity are the element counts of
 * gid/dist/sub_rowptr(-1) and sub_col: a pair whose rows would not fit is skipped, never written
 * out of bounds, and *overflow (device int32, may be NULL; sticky, the caller clears it) is set to 1
 * so that the host can tell a truncated batch from a complete one. */
int npi_khop_fill(const int32_t* rowptr, const int32_t* colm, int32_t num_nodes,
                  const int32_t* pairs, int32_t num_pairs, int32_t h, int32_t max_graph_nodes,
                  const int32_t* graph_ptr, const int32_t* edge_ptr,
                  int32_t* gid, uint8_t* dist, int32_t* sub_rowptr, int32_t* sub_col,
                  int32_t n_capacity, int32_t e_capacity, int32_t* overflow,
                  void* workspace, int64_t workspace_bytes, int32_t num_ctas, npi_stream_t stream);

/* Batch assembly on the device.  Replaces PyG Batch.from_data_list as used by DataLoader at
 * src/train_with_twoDataset.PY:142-143: picks B pairs (pair_index[b], or first+b if NULL) out
 * of the resident dataset arrays, gathers their targets/labels/cached counts and produces
 * graph_ptr for the input layer and the three pooled layers (k = ceil(ratio*n) in float32,
 * TopKPooling ratio rule), the input edge_ptr and sizes[8] = {N0,N1,N2,N3,E0,B,0,0}.
 * graph_ptrs is [4][B+1]. */
int npi_batch_prepare(const int32_t* pair_index, int32_t first, int32_t B,
                      const int32_t* pairs_all, const int32_t* y_all,
                      const int32_t* n_all, const int32_t* e_all, float ratio,
                      int32_t* pairs_b, int32_t* y_b, int32_t* graph_ptrs, int32_t* edge_ptr,
                      int32_t* sizes, npi_stream_t stream);

/* COO edge_index (int64 [2,E], rows src then dst, stride E) in SURVEY Appendix-B order from the
 * extractor's CSR: undirected edges in first-discovery order, (rna,prot) then (prot,rna).
 * Replaces the edge emission of src/classes.py:697-704 (whose order is Python set order).
 * local_ids != 0: per-graph local node ids (a PyG Data); else batch-global ids (a PyG Batch). */
int npi_subgraph_coo(const int32_t* graph_ptr, const int32_t* edge_ptr, int32_t B, int32_t h,
                     const int32_t* gid, const uint8_t* dist, const uint8_t* is_rna,
                     const int32_t* sub_rowptr, const int32_t* sub_col,
                     int64_t* edge_index, int64_t E_total, int32_t local_ids, npi_stream_t stream);

/* x[i] = [label | table[gid[i]]] materialised densely, [N,F] row-major.
 * Replaces src/classes.py:706-717,728 for callers that want Data.x. */
int npi_gather_features(const npi_features_t* feat, const int32_t* n_dev, int32_t n_host,
                        float* x_out, npi_stream_t stream);

/* Foreign COO -> CSR by destination (self loops dropped, per-row order = edge order).
 * Needed when SAGEConv/TopKPooling are called on a PyG-style edge_index (src/classes.py:62-71).
 * workspace >= npi_coo_to_csr_workspace_bytes(N,E). rowptr_out[N+1], col_out[E], count in rowptr_out[N]. */
int64_t npi_coo_to_csr_workspace_bytes(int32_t N, int64_t E);
int npi_coo_to_csr(const int64_t* edge_index, int64_t E, int32_t N,
                   int32_t* rowptr_out, int32_t* col_out,
                   void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Symmetry guard of a foreign edge_index: sums_out[0] / sums_out[1] (device uint64[2]) receive an
 * order-independent 64-bit fingerprint of the multiset {(src,dst)} and of its transpose {(dst,src)}
 * (self loops ignored).  They are equal iff the edge multiset is symmetric (up to a 2^-64 collision):
 * the reference's enclosing subgraphs always are (src/classes.py:697-704 emits both directions), and
 * the backward kernels rely on it (CSR^T = CSR); an asymmetric edge_index is rejected by the caller. */
int npi_edge_symmetry_sums(const int64_t* edge_index, int64_t E, uint64_t* sums_out, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * SAGEConv (torch-geometric 1.4.x: one weight [F,128] + bias, mean over neighbours U self).
 * Replaces self.convN(x, edge_index) + F.relu at src/classes.py:62,66,70 and, fused into the
 * epilogue, the TopKPooling score tanh(h.p/||p||) of src/classes.py:63,67,71.
 *   h_out[N,128] = act(mean_{j in row(i) U {i}} x_j . W + b)
 *   if pool_w: z_out[i] = h_i.pool_w / ||pool_w||, s_out[i] = tanh(z_i)
 * ------------------------------------------------------------------------------------------ */
int npi_sage_fwd(const npi_features_t* feat, const int32_t* rowptr, const int32_t* col,
                 const int32_t* n_dev, int32_t n_host,
                 const float* W, const float* b, int32_t relu,
                 const float* pool_w, float* h_out, float* z_out, float* s_out,
                 npi_stream_t stream);

/* Weight/bias gradient of SAGEConv from the (compact) pre-activation gradient:
 *   dW[F,128] = sum_r agg[sel[r]]^T dpre[r],  db = sum_r dpre[r]     (sel NULL = identity)
 * agg is recomputed from the inputs; partial sums are combined in a fixed order. */
int64_t npi_sage_bwd_weight_workspace_bytes(int32_t F);
int npi_sage_bwd_weight(const npi_features_t* feat, const int32_t* rowptr, const int32_t* col,
                        const int32_t* sel, const int32_t* nsel_dev, int32_t nsel_host,
                        const float* dpre, float* dW, float* db,
                        void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Input gradient of SAGEConv (F = 128):
 *   dx[j] = ( sum_{i in row(j) U {j}, new_id[i] >= 0} dpre[new_id[i]] / (deg_i+1) ) . W^T
 * (the edge set is symmetric so the transposed CSR is the CSR; new_id NULL = identity). */
int npi_sage_bwd_input(const float* dpre, const int32_t* new_id,
                       const int32_t* rowptr, const int32_t* col,
                       const int32_t* n_dev, int32_t n_host,
                       const float* W, float* dx, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Decomposed SAGEConv used by the fused engine.  By linearity mean(x).W = mean(x.W), so the
 * projection runs on the compact operand (feature table / pooled x') as a dense GEMM and the
 * CSR gather-reduce moves 128-wide rows only; the backward pass shares one transposed
 * aggregation (dxa) between the weight and the input gradient.  Same reference call sites as
 * npi_sage_fwd (src/classes.py:62,66,70); results agree with it to fp32 rounding.
 * ------------------------------------------------------------------------------------------ */
/* C[m,128] = A[m,K] . B   (B is [K,128]; transB != 0: B is [128,K] and used transposed) */
int npi_gemm_nn(const float* A, int32_t lda, const int32_t* m_dev, int32_t m_host, int32_t K,
                const float* B, int32_t transB, float* C, npi_stream_t stream);
/* Same product on the tcgen05 tensor cores (sm_100a): kind::tf32 MMAs with fp32 accumulators in
 * TMEM and the error-compensated 3xTF32 operand split (fp32-level accuracy).  A is streamed by TMA
 * (cp.async.bulk.tensor), the weights live in tensor memory.  K in 1..192 (transB: K in {32,64,96,128});
 * A and B 16-byte aligned, lda % 4 == 0; A must have at least m_host rows allocated (the tensor map
 * covers them; rows >= *m_dev are read but never stored).  single_pass bit 0: hi.hi product only
 * (plain TF32, diagnostic). */
int npi_gemm_nn_tc(const float* A, int32_t lda, const int32_t* m_dev, int32_t m_host, int32_t K,
                   const float* B, int32_t transB, float* C, int32_t single_pass, npi_stream_t stream);
/* out[K,128] = A[m,K]^T . D[m,128], rows split over CTAs, partials summed in a fixed order;
 * row0_partials (nullable, [R,128]) are added to out[0,:] (the structural-label row). */
int64_t npi_gemm_tn_workspace_bytes(int32_t K);
int npi_gemm_tn(const float* A, int32_t lda, const float* D, const int32_t* m_dev, int32_t m_host, int32_t K,
                const float* row0_partials, int32_t R, float* out,
                void* workspace, int64_t workspace_bytes, npi_stream_t stream);
/* out[K,128] = A[m,K]^T . D[m,128] on the tcgen05 tensor cores (3xTF32, fp32 TMEM accumulator,
 * both operands MN-major): rows split over one persistent CTA per SM, per-CTA partials summed in a
 * fixed order; K > 128 (the feature table of the layer-1 weight gradient) takes one pass per 128 columns
 * of A.  Columns K..lda-1 of A must be zero.  Same meaning of row0_partials as npi_gemm_tn. */
int64_t npi_gemm_tn_tc_workspace_bytes(void);
int npi_gemm_tn_tc(const float* A, int32_t lda, int32_t K, const float* D, const int32_t* m_dev, int32_t m_host,
                   const float* row0_partials, int32_t R, float* out, int32_t single_pass,
                   void* workspace, int64_t workspace_bytes, npi_stream_t stream);
/* h_i = act((sum_{j in row(i) U {i}} y_j)/(deg_i+1) + bias); y_j = Y[j] or, for the virtual input
 * layer (gid/dist non-NULL), Y[gid[j]] + dist[j]*w0 with Y the projected feature table and w0 the
 * label row of the weight.  Optional pooling score as in npi_sage_fwd. */
/* Rows of a CSR with more than 16 entries ("hub" rows: a protein that interacts with most of a
 * subgraph) are cut into segments of 32 entries, one warp each, so that no single warp walks a
 * 1000-entry row.  The segments are listed ONCE per CSR, when the CSR is produced (next to the
 * extraction / filter_adj), into hub_queue (counters, segment list, per-row arrival counters and
 * the buffer of partial sums; npi_hub_rows_bytes(e_max) bytes for a CSR of at most e_max entries);
 * the forward and the backward aggregation of that CSR both consume the list and leave the queue
 * ready for the next launch -- one launch at a time per queue.
 * Initialisation: the queue needs no zeroed memory.  npi_hub_rows_build (and npi_filter_adj after
 * npi_hub_rows_reset) writes the header, the segment list and every arrival counter a launch reads;
 * every launch rewinds the counters it used.  (16 and 32 are the shipped NPI_AG_HUB /
 * NPI_AG_SEG of csrc/hub.cuh.) */
int64_t npi_hub_rows_bytes(int64_t e_max);
/* row_order (nullable, 16 bytes per row, n_host rows): the rows with at most 16 entries BINNED BY
 * LENGTH CLASS -- {row, first entry, end, self payload} with self payload = gid[row] | dist[row] << 29
 * when gid/dist are given (virtual input layer), else the row id.  The 8-lane groups of a warp work in
 * lock step, so the pipelined aggregation kernels take four rows of the same class at a time; the
 * class totals live in the queue header (int32 hdr[4 + c] for classes c = 0..7: rows of 1, 2-3, 4-5,
 * 6-7, 8-11, 12-16 entries, whole-warp rows, hub rows; a row of 0 entries is class 0).  Class 6 holds
 * the rows of 17..NPI_AG_HUB entries and is empty at the shipped constants.  The order inside a class
 * is timing dependent and has no influence on any result (rows are independent). */
/* keep (nullable): only rows with keep[i] == i are listed -- the representative rows of npi_ctx_build: the
 * aggregation kernels then evaluate one row per layer-1 context and leave every other row of h/z/s untouched. */
int npi_hub_rows_build(const int32_t* rowptr, const int32_t* n_dev, int32_t n_host, int64_t e_max,
                       int32_t* hub_queue, int64_t hub_queue_bytes, const int32_t* gid, const uint8_t* dist,
                       void* row_order, const int32_t* keep, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Layer-1 contexts of a collated batch (csrc/ctx.cu).
 *   The reference's input row is a function of (global node id, hop label) alone
 *   (src/classes.py:706-717), so conv1 of src/classes.py:62 gives identical output rows for rows with the
 *   same (gid, label) and the same sequence of neighbour (gid, label): the subgraphs of a batch share
 *   their hubs, and ~4 of 5 rows repeat an earlier row's context.  rep_of[i] = the FIRST row of the batch
 *   with row i's context (rep_of[i] == i: a representative), found with a 64-bit hash over the packed
 *   entry stream of npi_entry_pack_virt and VERIFIED entry by entry (a colliding row stays its own
 *   representative).  stats (nullable, int32[4]): representatives, verification failures, entries in
 *   representative rows, 0.  Evaluating conv1 on the representatives only is bit-identical to the full
 *   evaluation (same summation order). */
/* label_sum (nullable, int32[n]): sum of the hop labels over a row's neighbours and the row itself (the coefficient of
 * the label column of conv1.weight in that row's aggregate). */
int64_t npi_ctx_workspace_bytes(int32_t n_max);
int npi_ctx_build(const int32_t* rowptr, const int32_t* packed, const int32_t* gid, const uint8_t* dist,
                  const int32_t* n_dev, int32_t n_host, int32_t* rep_of, int32_t* stats, int32_t* label_sum,
                  void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Stable LSD radix sort of (uint32 key, int32 value) pairs, key_bits low bits significant (csrc/sort.cu): the tool that
 * groups rows by context and (context, node) incidences by node in a FIXED order, so that the sums over a group are
 * reproducible without float atomics.  All n items are sorted; the result lands in (keys_a, vals_a) when
 * npi_sort_passes(key_bits) is even, else in (keys_b, vals_b). */
int64_t npi_sort_workspace_bytes(int64_t n_max);
int32_t npi_sort_passes(int32_t key_bits);
int npi_sort_pairs_u32(uint32_t* keys_a, int32_t* vals_a, uint32_t* keys_b, int32_t* vals_b, int64_t n, int32_t key_bits,
                       void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Per-context backward of conv1 (virtual input layer; replaces npi_pool_bwd phase 1 + npi_sage_aggregate_bwd +
 * npi_gid_reduce of that layer).  Rows of one context share h, z, s and the neighbour list, and the backward is linear in
 * the incoming gradient:  X_u = sum over the SELECTED member rows r of context u of (d_xp[new_id[r]] + readout terms),
 *   dU_u = relu'(h_u) (s_u X_u + (X_u . h_u)(1 - s_u^2) w/|w|),   G[v] = sum_{u : v in N(u) U {u}} dU_u / (deg_u + 1).
 * Index structures, built once per batch next to the extraction (npi_ctx_index_build):
 *   class_keys/class_rows [n_host]: rows sorted by representative (members ascending; padding rows carry key n_host); the
 *     result is in the _b pair when npi_ctx_class_result_in_b(n_host) != 0;
 *   class_ptr2 [n_host+1], class_rep [n_host], *n_ctx: contexts numbered by ascending representative row; context u owns
 *     the entries [class_ptr2[u], class_ptr2[u+1]) of a CSR with TWO entries per member (npi_ctx_class_pack);
 *   inv_ptr [V+1], inv_sel [n_host + e_max] int32 pairs: CSR by global node id over the (context, node) incidences,
 *     entries {context, bits of 1/(deg+1)} (unused tail entries {-1, 0}).
 * Per step: npi_ctx_scatter_max adds the max-readout gradient into its argmax rows of d_xp (each (row, column) at most
 * once: no atomics); npi_ctx_class_pack fills the class CSR's entries {row of d_xp, 1}, {mean-readout row of the member's
 * graph, 1/k} -- the readout gradient [B,256] must live in the SAME buffer as d_xp, readout_row0 rows behind its start --;
 * npi_csr_gather_sum (the transposed-aggregation kernel, no self term) sums them into X; npi_ctx_finish turns X into dU in
 * place and leaves per-CTA partials in npi_pool_bwd's layout (npi_pool_bwd(phases = 2) finishes d_pool_w / d_bias; needs
 * npi_ctx_finish_partials() == the number npi_pool_bwd uses) plus label_partials [npi_ctx_finish_partials()][128]
 * (label row of conv1.weight); npi_csr_gather_sum over inv_ptr/inv_sel then gives G. */
int64_t npi_ctx_index_workspace_bytes(int32_t n_max, int64_t e_max);
int32_t npi_ctx_class_result_in_b(int32_t n_max);
int npi_ctx_index_build(const int32_t* rowptr, const int32_t* packed, const int32_t* gid, const int32_t* rep_of,
                        const int32_t* n_dev, int32_t n_host, int64_t e_max, int32_t V,
                        uint32_t* class_keys_a, int32_t* class_rows_a, uint32_t* class_keys_b, int32_t* class_rows_b,
                        int32_t* class_ptr2, int32_t* class_rep, int32_t* n_ctx,
                        int32_t* inv_ptr, void* inv_sel, void* workspace, int64_t workspace_bytes, npi_stream_t stream);
int npi_ctx_class_pack(const int32_t* class_rows, const int32_t* n_dev, int32_t n_host, const int32_t* new_id,
                       const int32_t* batch_out, const int32_t* graph_ptr_out, int32_t readout_row0, void* class_sel,
                       npi_stream_t stream);
int npi_ctx_scatter_max(const float* d_readout, const int32_t* argmax, int32_t B, float* d_xp, npi_stream_t stream);
int32_t npi_ctx_finish_partials(void);
int npi_ctx_finish(float* XU, const int32_t* class_rep, const int32_t* n_ctx_dev, int32_t n_ctx_host, const float* h,
                   const float* z, const float* s, const float* pool_w, int32_t relu, const int32_t* rowptr,
                   const int32_t* label_sum, float* label_partials, void* workspace, int64_t workspace_bytes,
                   npi_stream_t stream);
/* out[r] = sum over the packed entries {row, weight bits} of CSR row r of src[row] * weight (entries with row < 0 are
 * skipped): npi_sage_aggregate_bwd's pipelined kernel without the self term, on any CSR whose hub queue / binned row
 * order npi_hub_rows_build made. */
int npi_csr_gather_sum(const float* src, const int32_t* rowptr, const void* packed, int32_t n_rows, float* out,
                       int32_t* hub_queue, const void* row_order, npi_stream_t stream);

/* Packed entry streams of a CSR (one value per CSR entry, in CSR order), built once per CSR off the
 * critical path so that the aggregation kernels read ONE coalesced value per entry instead of
 * chasing col -> gid/dist (virtual input layer) or col -> new_id, rowptr[i], rowptr[i+1] (backward):
 *   npi_entry_pack_virt : packed[k] = gid[col[k]] | dist[col[k]] << 29          (int32; V < 2^29)
 *   npi_entry_pack_sel  : packed[k] = { new_id[col[k]] (or col[k] if new_id NULL),
 *                                       bits of 1/(deg_col+1), 0 if not selected }  (int32 pair)
 * e_max = capacity of `packed` in entries; the realised count rowptr[n] is read on the device. */
int npi_entry_pack_virt(const int32_t* rowptr, const int32_t* col, const int32_t* gid, const uint8_t* dist,
                        const int32_t* n_dev, int32_t n_host, int32_t V, int64_t e_max, int32_t* packed,
                        npi_stream_t stream);
int npi_entry_pack_sel(const int32_t* rowptr, const int32_t* col, const int32_t* new_id, const int32_t* n_dev,
                       int32_t n_host, int64_t e_max, void* packed, npi_stream_t stream);
/* pipelined != 0: rows taken in the length-class order `row_order` of npi_hub_rows_build, software
 * pipelined (row records two iterations ahead, first entries one ahead); for the virtual input layer
 * it reads `packed` (npi_entry_pack_virt) instead of col/gid/dist.
 * pipelined == 0: rows in index order, plain dependent chain (packed / row_order ignored).
 * Results are bit-identical. */
int npi_sage_aggregate_fwd(const float* Y, const int32_t* gid, const uint8_t* dist, const float* w0,
                           const int32_t* rowptr, const int32_t* col, const int32_t* n_dev, int32_t n_host,
                           const float* bias, int32_t relu, const float* pool_w,
                           float* h, float* z, float* s, int32_t* hub_queue, const int32_t* packed,
                           const void* row_order, int32_t pipelined, npi_stream_t stream);
/* dxa[j] = sum_{i in row(j) U {j}, new_id[i] >= 0} dpre[new_id[i]] / (deg_i+1)   (new_id NULL = identity).
 * packed non-NULL (npi_entry_pack_sel of this CSR and new_id; needs row_order): the pipelined kernel;
 * NULL: the plain one. */
int npi_sage_aggregate_bwd(const float* dpre, const int32_t* new_id, const int32_t* rowptr, const int32_t* col,
                           const int32_t* n_dev, int32_t n_host, float* dxa,
                           int32_t* hub_queue, const void* packed, const void* row_order, npi_stream_t stream);
/* Occurrence lists of the batch nodes by global serial (int only, deterministic): occ_ptr[V+1],
 * occ_node[N] sorted ascending inside every list.  Built once per batch next to the extraction. */
int64_t npi_gid_index_workspace_bytes(int32_t num_nodes, int32_t n_max);
int npi_gid_index_build(const int32_t* gid, const int32_t* n_dev, int32_t n_host, int32_t num_nodes,
                        int32_t* occ_ptr, int32_t* occ_node, void* workspace, int64_t workspace_bytes,
                        npi_stream_t stream);
/* G[v] = sum_{j in list(v)} dxa[j]  and per-CTA partials of sum_j dist[j]*dxa[j] (label row of the
 * layer-1 weight gradient); label_partials is [npi_gid_reduce_partials(), 128]. */
int32_t npi_gid_reduce_partials(void);
int npi_gid_reduce(const float* dxa, const uint8_t* dist, const int32_t* occ_ptr, const int32_t* occ_node,
                   int32_t num_nodes, float* G, float* label_partials, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * TopKPooling(128, ratio) -- src/classes.py:49,51,53 / calls :63,67,71 (PyG 1.4.2 semantics,
 * SURVEY Appendix A.3).
 * ------------------------------------------------------------------------------------------ */
/* score only (module API; the fused path gets it from npi_sage_fwd) */
int npi_topk_score(const float* h, const int32_t* n_dev, int32_t n_host, const float* pool_w,
                   float* z_out, float* s_out, npi_stream_t stream);
/* per-graph selection: keep graph_ptr_out[g+1]-graph_ptr_out[g] highest scores, descending,
 * ties -> lower node index.  perm[N'] (old ids), new_id[N] (-1 = dropped), batch_out[N'].
 * max_graph_nodes = host upper bound of the largest graph (sizes the sort).
 * Bit-exact integer outputs for given scores.
 * row_map (nullable, with perm_src): the score of row i is s[row_map[i]] (rows that share a layer-1
 * context, npi_ctx_build, keep one copy of h/z/s at their representative) and perm_src[r] =
 * row_map[perm[r]] -- the row the gating and the pooling backward read h/z/s from. */
int64_t npi_topk_select_workspace_bytes(int32_t B, int32_t max_graph_nodes);
int npi_topk_select(const float* s, const int32_t* graph_ptr_in, const int32_t* graph_ptr_out,
                    int32_t B, int32_t max_graph_nodes,
                    int32_t* perm, int32_t* new_id, int32_t* batch_out,
                    const int32_t* row_map, int32_t* perm_src,
                    void* workspace, int64_t workspace_bytes, npi_stream_t stream);
/* xp[r] = h[perm[r]] * s[perm[r]]; per-graph readout [max | mean] (gmp/gap + cat,
 * src/classes.py:64,68,72) written (accumulate=0) or added (accumulate=1, the x1+x2+x3 of
 * src/classes.py:74) into readout[B,256]; argmax[B,128] = row (new numbering) of the max.
 * phases: 0 = everything; 1 = xp + per-range partial max/sum/argmax (left in the workspace);
 * 2 = readout / argmax from the partials of an earlier phase-1 call on the SAME workspace. */
int64_t npi_pool_gate_readout_workspace_bytes(int32_t B);
int npi_pool_gate_readout(const float* h, const float* s, const int32_t* perm,
                          const int32_t* graph_ptr_out, int32_t B,
                          float* xp, float* readout, int32_t accumulate, int32_t* argmax,
                          void* workspace, int64_t workspace_bytes, int32_t phases, npi_stream_t stream);
/* filter_adj on CSR: new row r = old row perm[r] with dropped sources removed and the rest
 * relabelled, order preserved.  rowptr_out[N'+1], col_out[<= E]; edge count in rowptr_out[N'].
 * hub_queue / row_order (nullable; hub_e_max = the entry capacity the queue was sized for): the hub queue and the binned
 * row order of the NEW CSR are produced on the way (a row's segments need only its length, its record only its final
 * extent) -- what npi_hub_rows_build would do in two more kernels on the chain the next aggregation waits for.  The
 * caller zeroes the queue header first (npi_hub_rows_reset, any time after the queue's last consumer). */
int64_t npi_filter_adj_workspace_bytes(int32_t n_new_max);
int npi_filter_adj(const int32_t* rowptr, const int32_t* col, const int32_t* perm,
                   const int32_t* new_id, const int32_t* nnew_dev, int32_t nnew_host,
                   int32_t* rowptr_out, int32_t* col_out,
                   int32_t* hub_queue, int64_t hub_e_max, void* row_order,
                   void* workspace, int64_t workspace_bytes, npi_stream_t stream);
int npi_hub_rows_reset(int32_t* hub_queue, npi_stream_t stream);
/* filter_adj on a COO edge_index (operator API: TopKPooling returns edge_index', src/classes.py:63):
 * keeps edge e iff both endpoints survive, relabels through new_id, preserves order.  out is
 * int64 [2,E] (row stride E); the kept count lands in *count_dev. */
int64_t npi_filter_edges_coo_workspace_bytes(int64_t E);
int npi_filter_edges_coo(const int64_t* edge_index, int64_t E, const int32_t* new_id, int64_t* out,
                         int32_t* count_dev, void* workspace, int64_t workspace_bytes, npi_stream_t stream);
/* Backward of global_max_pool / global_mean_pool (operator API, src/classes.py:64,68,72):
 * dx[r] = d_readout[g, 128:]/k_g (use_mean) + [argmax[g,c] == r] d_readout[g, :128] (use_max). */
int npi_readout_bwd(const float* d_readout, const int32_t* argmax, const int32_t* graph_ptr, const int32_t* batch,
                    int64_t n, int32_t use_max, int32_t use_mean, float* dx, npi_stream_t stream);
/* Backward of readout + gating + score + ReLU for one layer.  Inputs: d_xp[N',128] (gradient
 * w.r.t. the pooled features coming from the next SAGEConv; NULL = 0), d_readout[B,256]
 * (gradient of the summed readout), saved h, z, s, perm, batch', argmax, graph_ptr_out.
 * Outputs: dpre[N',128] (compact pre-activation gradient of the selected rows),
 * d_pool_w[128], and (nullable) d_bias[128] = sum_r dpre[r], the SAGEConv bias gradient.
 * relu != 0 applies the ReLU mask (h > 0).
 * phases: 0 = everything; 1 = dpre + the per-CTA partial sums (left in the workspace); 2 = d_pool_w /
 * d_bias from the partials of an earlier phase-1 call on the SAME workspace (only the optimizer
 * waits for them: the engine runs phase 2 on its auxiliary stream, one workspace per layer). */
int64_t npi_pool_bwd_workspace_bytes(void);
int npi_pool_bwd(const float* d_xp, const float* d_readout, const float* h, const float* z,
                 const float* s, const int32_t* perm, const int32_t* batch_out,
                 const int32_t* argmax, const int32_t* graph_ptr_out,
                 const int32_t* nnew_dev, int32_t nnew_host, int32_t B,
                 const float* pool_w, int32_t relu, float* dpre, float* d_pool_w, float* d_bias,
                 void* workspace, int64_t workspace_bytes, int32_t phases, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * MLP head + loss: src/classes.py:55-57,74-80 and F.nll_loss at src/train_with_twoDataset.PY:53.
 * params: lin1 [128,256]+[128], lin2 [64,128]+[64], lin3 [2,64]+[2] (torch.nn.Linear layout).
 * Dropout p=0.5 (training != 0): mask from Philox4x32-10 keyed by (seed; sample id, feature,
 * *step_dev) -- sample id = sample_ids[b] or sample_id_base+b, so 1-GPU and N-GPU runs draw the
 * same mask for the same sample -- or, if drop_mask_in != NULL, the injected uint8 mask [B,128]
 * (1 = keep).  step_dev (nullable) is a device counter so a replayed CUDA graph draws fresh masks.
 * Saves a1[B,128] (after ReLU+dropout), a2[B,64], logp[B,2], drop_mask_out[B,128].
 * loss_out[0] = sum_b -logp[b][y_b] * loss_scale  (loss_scale = 1/B_global), y NULL = no loss.
 * phases: 0 = everything; 1 = the MLP (a1, a2, logp, mask); 2 = only the loss from logp.
 * ------------------------------------------------------------------------------------------ */
int npi_head_fwd(const float* readout, int32_t B,
                 const float* w1, const float* b1, const float* w2, const float* b2,
                 const float* w3, const float* b3,
                 int32_t training, const uint8_t* drop_mask_in, uint64_t seed, const int32_t* step_dev,
                 const int32_t* sample_ids, int32_t sample_id_base,
                 const int32_t* y, float loss_scale,
                 float* a1, uint8_t* drop_mask_out, float* a2, float* logp, float* loss_out,
                 int32_t phases, npi_stream_t stream);
/* backward: gradients of the six head tensors and d_readout[B,256]; workspace >= B*194 floats.
 * phases: 0 = everything; 1 = only the per-sample deltas (workspace) and d_readout -- what the layers
 * below wait for; 2 = only the six weight gradients from the deltas of an earlier phase-1 call (only
 * the optimizer waits for them, so the engine runs this on its auxiliary stream).
 * Upstream gradient: d_logp[B,2] if non-NULL (what autograd hands to the op), else the mean-NLL
 * gradient (softmax - onehot(y)) * loss_scale. */
/* Training step: npi_head_fwd(phases = 1) and npi_head_bwd(phases = 1) of the mean-NLL loss in ONE launch (the CTA that
 * computed a sample's activations still holds them): a1, drop mask, a2, logp as npi_head_fwd; per-sample deltas into the
 * workspace and d_readout [B,256] as npi_head_bwd(phases = 1) -- bit-identical to the two calls.  The scalar loss and the
 * weight gradients remain npi_head_fwd(phases = 2) / npi_head_bwd(phases = 2)
 * (src/classes.py:74-80, src/train_with_twoDataset.PY:53-54). */
int npi_head_fwd_delta(const float* readout, int32_t B, const float* w1, const float* b1, const float* w2,
                       const float* b2, const float* w3, const float* b3, int32_t training,
                       const uint8_t* drop_mask_in, uint64_t seed, const int32_t* step_dev,
                       const int32_t* sample_ids, int32_t sample_id_base, const int32_t* y, float loss_scale,
                       float* a1, uint8_t* drop_mask_out, float* a2, float* logp, float* d_readout,
                       void* workspace, int64_t workspace_bytes, npi_stream_t stream);
int64_t npi_head_bwd_workspace_bytes(int32_t B);
int npi_head_bwd(const float* readout, int32_t B,
                 const float* w1, const float* w2, const float* w3,
                 const float* a1, const uint8_t* drop_mask, const float* a2, const float* logp,
                 const int32_t* y, float loss_scale, const float* d_logp,
                 float* d_w1, float* d_b1, float* d_w2, float* d_b2, float* d_w3, float* d_b3,
                 float* d_readout, void* workspace, int64_t workspace_bytes, int32_t phases, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer: torch.optim.Adam(lr, weight_decay) with L2-in-gradient
 * (src/train_with_twoDataset.PY:130; Appendix A.6) over flat buffers.  lr_dev (float) and
 * step_dev (int32) live in DEVICE
 * memory so a captured CUDA graph can be replayed while the host changes lr.  *step_dev is the
 * number of completed steps; the call performs step *step_dev+1 and then increments it.
 * grad_scale multiplies the gradient first (1/world_size after a sum all-reduce).
 * ------------------------------------------------------------------------------------------ */
int npi_adam_l2_step(float* params, const float* grads, float* m, float* v, int64_t n,
                     float* lr_dev, int32_t* step_dev, float beta1, float beta2, float eps,
                     float weight_decay, float grad_scale, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Data-parallel gradient exchange fused with the optimizer (SURVEY.md 8e / 8b
 * "npi_allreduce_adam_fused").  The reference trains on one device
 * (src/train_with_twoDataset.PY:46-57: loss.backward(); optimizer.step()); with one process per
 * GPU the step's only exchange is the sum of the flat gradient buffer.  Each rank owns ONE peer
 * buffer = [header of npi_peer_header_bytes() | n floats of gradients] that the other ranks map
 * over NVLink (cudaIpc).  These four calls are the library's only allocating / mapping calls
 * (IPC handles need a cudaMalloc'ed base); they are host-synchronous set-up, never on a stream.
 *   npi_peer_alloc : cudaMalloc + zero `bytes`, export the 64-byte IPC handle.
 *   npi_peer_open  : map a peer's handle (lazy peer access), npi_peer_close unmaps it,
 *   npi_peer_free  : release the own buffer.
 * npi_allreduce_adam_fused (ONE kernel, asynchronous, graph-capturable, no host involvement):
 *   publishes "gradients of this step complete" to every peer, waits for every peer, sums the
 *   `world` gradient buffers read from peer memory in RANK ORDER (bit-identical on all ranks, no
 *   float atomics), applies npi_adam_l2_step's update to the replicated params/m/v, then
 *   exchanges "done reading" flags so the local buffer may be overwritten when the kernel exits
 *   (closing != 0).  grads_offset (floats, multiple of 4) selects the gradient buffer inside every rank's
 *   peer allocation: a caller that ALTERNATES two buffers from step to step passes closing = 0 -- a peer's
 *   arrival at step e+1 implies it finished reading step e, and the buffer of step e is next written at
 *   step e+2 -- and calls npi_peer_barrier before it ever uses the same buffer twice in a row.
 *   peer_base_h[world]: HOST array of the mapped base pointers (entry `rank` = own buffer).
 *   state[4] uint32 device words, zero-initialised once: exchanges completed, block counter,
 *   status (1 = a wait exceeded timeout_ms -- the step's result is invalid), reserved.
 *   *step_dev is incremented like npi_adam_l2_step does.
 * npi_peer_barrier: all ranks meet (one tiny kernel; flag words of the closing handshake, counter state[3]).
 * ------------------------------------------------------------------------------------------ */
int64_t npi_peer_header_bytes(void);
int npi_peer_alloc(int64_t bytes, void** dev_ptr_h, unsigned char* ipc_handle_h);
int npi_peer_open(const unsigned char* ipc_handle_h, void** dev_ptr_h);
int npi_peer_close(void* dev_ptr);
int npi_peer_free(void* dev_ptr);
int npi_allreduce_adam_fused(const void* const* peer_base_h, int32_t world, int32_t rank,
                             float* params, float* m, float* v, int64_t n,
                             float* lr_dev, int32_t* step_dev, uint32_t* state,
                             float beta1, float beta2, float eps, float weight_decay,
                             float grad_scale, int32_t timeout_ms, int64_t grads_offset, int32_t closing,
                             npi_stream_t stream);
int npi_peer_barrier(const void* const* peer_base_h, int32_t world, int32_t rank, uint32_t* state, int32_t timeout_ms,
                     npi_stream_t stream);

/* out[K,128] = table[:, :K]^T . G (+ sum_r row0_partials[r] on row 0) for a SMALL table (V rows, thousands): the layer-1
 * weight gradient d conv1.weight of the virtual input layer (src/classes.py:62 through the feature table) in two
 * launches, fixed summation order.  Large tables use npi_gemm_tn_tc. */
int64_t npi_table_grad_workspace_bytes(int32_t K);
int npi_table_grad(const float* table, int32_t lda, int32_t K, const float* G, int32_t V, const float* row0_partials,
                   int32_t R, float* out, void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Tuning aid: buf[idx] (uint64) = %globaltimer when the stream reaches this point (one 1-thread kernel). */
int npi_debug_stamp(void* buf, int32_t idx, npi_stream_t stream);

/* acc[0] += a * x[0] on the device: the epoch-loss accumulator `loss_all += data.num_graphs * loss.item()` of
 * src/train_with_twoDataset.PY:55 without the host round trip (one launch, capturable). */
int npi_scalar_axpy(float* acc, const float* x, float a, npi_stream_t stream);

/* Confusion counts of src/methods.py:87-127: pred = argmax(logp), counts[4] += {TP,FN,TN,FP}
 * (int64, device).  threshold < 0: argmax rule; else positive iff exp(logp[:,1]) > threshold
 * (src/case_study_negativeSample.py:235-253). */
int npi_confusion_counts(const float* logp, const int32_t* y, int32_t B, float threshold,
                         int64_t* counts, npi_stream_t stream);

/* Ranking metrics of n scored pairs (csrc/rank.cu): the threshold-free evaluation next to the confusion matrix of
 * src/methods.py:87-127 -- the ROC AUC and PR summaries the reference's src/compare_withKmer_noKmer.py:39-74,213-368
 * computes with sklearn from saved checkpoints.  The semantics are sklearn's (_binary_clf_curve, roc_curve,
 * roc_auc_score, average_precision_score, precision_recall_curve, auc):
 *  - the distinct scores in descending order are the thresholds r = 0 .. n_thresholds-1; -0.0 and +0.0 are one
 *    threshold, +-inf are ordinary scores.  A NaN score sets status bit 0, a label other than 0 or 1 sets bit 1 (the
 *    other outputs are then meaningless).
 *  - tps[r] / fps[r] = labels 1 / labels 0 with score >= threshold r (cumulative): thresholds, fps / n_neg, tps / n_pos
 *    equal roc_curve(y, s, drop_intermediate=False) without its leading inf point.
 *  - twice_u = sum_r (fps[r] - fps[r-1]) * (tps[r] + tps[r-1]), tps[-1] = fps[-1] = 0: exact, twice the Mann-Whitney U
 *    with ties counted one half; ROC AUC = twice_u / (2 n_pos n_neg).  twice_u < n^2 / 2 fits int64.
 *  - areas[0] = average precision = sum_r (tps[r] - tps[r-1]) * tps[r] / (tps[r] + fps[r]) / n_pos (fp64).
 *  - areas[1] = trapezoidal area under precision_recall_curve's points, its end point (recall 0, precision 1)
 *    included: auc(recall, precision).
 * summary (int64[4]) = {n_pos, n_neg, n_thresholds, twice_u}.  thresholds / tps / fps (nullable each) receive the curve
 * in their first n_thresholds entries (n entries each).  1 <= n < 2^31.  Every output is bit-identical on reruns and
 * under any permutation of the input (only run ends of the sorted scores are read; no float atomics).  17 launches, no
 * host synchronisation; the workspace needs no initialisation. */
int64_t npi_rank_workspace_bytes(int64_t n_max);
int npi_rank_curve(const float* scores, const int32_t* labels, int64_t n, int64_t* summary, double* areas,
                   float* thresholds, int32_t* tps, int32_t* fps, int32_t* status,
                   void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Top-k items of every group by score (csrc/topk.cu): the per-node ranking of a scoring sweep that the reference's
 * case studies (src/case_study_negativeSample.py, src/case_study.py) read -- for an RNA its most likely protein
 * partners, for a protein its most likely RNAs.
 *  - item i (0 <= i < n) has score scores[i] and group group[i], 0 <= group[i] < num_groups.
 *  - for every group g the first out_count[g] = min(k, |g|) entries of row g of out_pos / out_score ([num_groups, k],
 *    row-major) are the items of g ranked by descending score; ties break by ascending i.  -0.0 and +0.0 are one value
 *    (their order comes from i, not from the sign); +-inf are ordinary scores.  out_score is the input value, copied
 *    bit for bit.  Entries past out_count[g] are out_pos = -1 and out_score = NaN; an empty group has out_count 0.
 *  - status (int32[1]): bit 0 = a NaN score, bit 1 = a group id out of range; when either is set the other outputs are
 *    meaningless.
 * 1 <= k <= 1024, 1 <= n < 2^31, 1 <= num_groups < 2^24.  Outputs are bit-identical on reruns (no float atomics).
 * 3 + 3 * npi_sort_passes(ceil(log2 num_groups)) launches (6 up to 512 groups, 9 up to 262,144, else 12), no host
 * synchronisation, capturable in a CUDA graph; the workspace needs no initialisation. */
int64_t npi_group_topk_workspace_bytes(int64_t n_max, int32_t num_groups);
int npi_group_topk(const float* scores, const int32_t* group, int64_t n, int32_t num_groups, int32_t k,
                   int32_t* out_pos, float* out_score, int32_t* out_count, int32_t* status,
                   void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Filtered rank of every held-out interaction among its group's candidates (csrc/grouprank.cu): MRR, Hits@K and the
 * per-group ROC AUC of a scoring sweep -- for each RNA, where its true partners rank among all the proteins it could
 * pair with, and for each protein among its RNAs (the question of the reference's src/case_study.py and
 * src/case_study_negativeSample.py, and the link-prediction reading of them).
 *  - inputs: scores float32[n]; labels int32[n], 1 = query (a held-out interaction), 0 = competitor (a sampled negative
 *    or an unlabelled candidate pair); group int32[n], 0 <= group < num_groups; hits_k: HOST array of n_hits int32,
 *    1 <= n_hits <= 8, every K >= 1.
 *  - per query i of group g: above_i = competitors of g with a score strictly greater than s_i, tied_i = competitors of g
 *    with a score equal to s_i.  Scores compare as rank_key does: -0.0 and +0.0 are equal, +-inf are ordinary scores.
 *    The other queries of g never compete (the filtered setting).
 *  - rank_i = above_i + tied_i / 2 + 1, the mean of the optimistic rank above + 1 and the pessimistic rank
 *    above + tied + 1 (ties get half credit, as in OGB's MRR).  Comparisons use 2 rank = 2 above + tied + 2 in integers;
 *    1 / rank is computed in fp64.
 *  - per group (device, num_groups entries each): n_pos, n_neg (int32); twice_u (int64) = sum over the queries of g of
 *    2 (n_neg[g] - above_i - tied_i) + tied_i.  twice_u / (2 n_pos n_neg) equals sklearn's roc_auc_score on the group's
 *    items.
 *  - summary (device int64[3 + n_hits]) = {n_queries, n_unranked, n_groups_scored, hits[0 .. n_hits-1]}: n_queries =
 *    queries whose group has at least one competitor (the ranked queries); n_unranked = queries in groups without a
 *    competitor, left out of MRR and Hits (their counts are 0 / 0); n_groups_scored = groups with both classes;
 *    hits[h] = ranked queries with 2 above + tied + 2 <= 2 K_h.  sum_rr (device double[1]) = sum of 1 / rank over the
 *    ranked queries.
 *  - above / tied (nullable each, int32[n], input order): the counts of every query, -1 for competitors.
 *  - status (int32[1]): bit 0 = a NaN score, bit 1 = a label other than 0 or 1, bit 2 = a group id out of range; when any
 *    bit is set the other outputs are meaningless.
 * 1 <= n < 2^31, 1 <= num_groups < 2^24.  Every output is bit-identical on reruns and under any permutation of the input
 * (the per-item outputs follow their items): each tie run of (group, score) contributes one term npos_run / rank at its
 * run end, whose sorted index does not depend on the input order; no float atomics.  21 + 3 *
 * npi_sort_passes(ceil(log2 num_groups)) launches (24 up to 512 groups, 27 up to 262,144, else 30), no host
 * synchronisation, capturable in a CUDA graph; the workspace needs no initialisation. */
int64_t npi_group_rank_workspace_bytes(int64_t n_max, int32_t num_groups);
int npi_group_rank(const float* scores, const int32_t* labels, const int32_t* group, int64_t n, int32_t num_groups,
                   const int32_t* hits_k, int32_t n_hits, int32_t* n_pos, int32_t* n_neg, int64_t* twice_u,
                   int64_t* summary, double* sum_rr, int32_t* above, int32_t* tied, int32_t* status,
                   void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* Input attribution of scored pairs (csrc/attrib.cu): why the model scores a pair as it does, in terms of the nodes and
 * the input features of its enclosing subgraph -- the follow-up question to the case-study ranking of the reference's
 * src/case_study.py and src/case_study_negativeSample.py (which proteins does this lncRNA interact with, and why).
 *  - for a pair p let t(p) be its target: logp[p, c] for a class c, or p_c = exp(logp[p, c]).  The network runs in
 *    evaluation mode (no dropout), exactly the forward the scoring sweep runs.  Every discrete decision is the one that
 *    forward took (top-k selections, ReLU masks, the row global_max_pool routes to): the usual piecewise gradient.
 *  - row i of p's subgraph has the layer-1 input x_i of width F: x_i[0] = (float)dist[i] (the structural label),
 *    x_i[c] = table[gid[i] * ld + c] for 1 <= c < F (npi_features_t, virtual form).
 *  - input: dxa [n_rows, 128] (16-byte aligned), the gradient of the batch's targets with respect to the projected
 *    layer-1 rows x_i . W1 -- what the backward pass leaves after the transposed layer-1 aggregation
 *    (npi_sage_aggregate_bwd, or npi_tiny_bwd phase 1 on the small-subgraph path) when it is seeded with
 *    d_logp[b] = e_c (or p_c e_c) for every pair b.  Subgraphs are disjoint row ranges and nothing in evaluation mode
 *    couples the pairs of a batch, so one backward pass gives every pair its own gradient.  It must be per row: the
 *    per-context backward of conv1 (npi_csr_gather_sum over contexts) sums rows of different subgraphs.
 *  - w1 = conv1.weight [F, 128] row-major; graph_ptr [B + 1] = rows of pair b at the input layer (npi_batch_prepare).
 *  - outputs: grad_x[i][c] = d t(p) / d x_i[c] = (dxa_i . W1^T)[c]  ([n_rows, F] row-major; NULL = not written);
 *             node_attr[i] = sum_c x_i[c] grad_x[i][c]  (gradient x input per row);
 *             feature_attr[p][c] = sum over the rows i of p of x_i[c] grad_x[i][c]  ([B, F] row-major).
 *    The rows used are those below min(n_rows, graph_ptr[B]); n_rows (host) sizes the grid and the workspace.
 * 1 <= F <= 256, B >= 1, n_rows >= 0, ld >= F.  SIMT fp32 (the backward pass before it costs far more).  Every sum has
 * a fixed order: a pair's rows are summed in chunks of 32 counted from its first row, and a pair of several chunks adds
 * their partials in chunk order (a CTA per pair), so the outputs are bit-identical on reruns and a pair's sums do not
 * depend on where it sits in its batch.  No float atomics, no host synchronisation, three launches (two when n_rows is
 * 0); the workspace (npi_input_attribution_workspace_bytes) needs no initialisation. */
int64_t npi_input_attribution_workspace_bytes(int32_t n_rows, int32_t B, int32_t F);
int npi_input_attribution(const float* dxa, const int32_t* gid, const uint8_t* dist, const int32_t* graph_ptr, int32_t B,
                          int32_t n_rows, const float* table, int32_t ld, int32_t F, const float* w1,
                          float* node_attr, float* feature_attr, float* grad_x,
                          void* workspace, int64_t workspace_bytes, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * node2vec on the GPU (the stage that produces the embedding columns of the feature table).
 * Replaces node2vec-master/src/node2vec.py and main.py:78-92 of the reference over a CSR with
 * SORTED adjacency (rowptr[V+1], col[E] int32; weight[E] float64 or NULL = unit weights, what
 * main.py:read_graph :63-76 builds for the unweighted default).
 *
 * npi_n2v_etab_scan: etab_ptr[e] = sum_{e'<e} deg(col[e']), etab_ptr[E] = total slots of all
 *   second-order tables (int64, device).
 * npi_n2v_alias_tables: preprocess_transition_probs + get_alias_edge + alias_setup
 *   (node2vec.py:55-134).  Node table of v at nodeJ/nodeq + rowptr[v]; edge table of CSR entry e
 *   (src -> col[e]) at edgeJ/edgeq + etab_ptr[e], deg(col[e]) slots.  q is float64 and bit-equal to
 *   the reference's numpy array.  work: E + etab_total int32 of scratch.
 * npi_n2v_alias_from_probs: alias_setup (node2vec.py:107-134) of one given distribution
 *   (probs[K] float64); work: K int32.
 * npi_n2v_walks: simulate_walks / node2vec_walk (node2vec.py:13-53).  Walk w (0 <= w < num_walks)
 *   starts at starts[w % num_starts] and draws step s from Philox4x32-10(counter = (walk_id0 + w,
 *   s, 0, 0), key = seed).  walks[num_walks, walk_length] (unused tail = -1), lens[num_walks].
 * npi_n2v_vocab_count: counts[v] += occurrences of v in the walks (int64; the caller zeroes it).
 * npi_n2v_init_vectors: syn0[v][c] = (u - 0.5)/dim (word2vec's initial vectors), u from Philox.
 * npi_n2v_skipgram: one epoch of skip-gram with negative sampling over the walks
 *   (main.py:87 Word2Vec(sg=1, window, negative=5, min_count=0)): keep[V] = frequent-word keep
 *   probability, (negJ, negq) = alias table of the count^0.75 distribution, learning rate of walk w
 *   = max(min_alpha, alpha - (alpha - min_alpha) * tok_before[w] / total_tokens).
 *   schedule 1: ONE warp, pair-at-a-time order (deterministic).  schedule 0: a warp per walk, lock-free
 *   plain stores ("hogwild", like gensim's worker threads).  schedule 2: a warp per walk, row updates as
 *   vector float atomic adds (no lost update).  Schedules 0 and 2 are the one place in this library whose
 *   result depends on scheduling.  max_warps > 0 caps the number of concurrent walks.
 * ------------------------------------------------------------------------------------------ */
int npi_n2v_etab_scan(const int32_t* rowptr, const int32_t* col, int32_t V, int64_t E, int64_t* etab_ptr,
                      npi_stream_t stream);
int npi_n2v_alias_tables(const int32_t* rowptr, const int32_t* col, const double* weight, int32_t V, int64_t E,
                         double p, double q, const int64_t* etab_ptr, int32_t* nodeJ, double* nodeq,
                         int32_t* edgeJ, double* edgeq, int32_t* work, int64_t work_elems, int64_t etab_total,
                         npi_stream_t stream);
int npi_n2v_alias_from_probs(const double* probs, int32_t K, int32_t* J, double* q, int32_t* work,
                             npi_stream_t stream);
int npi_n2v_walks(const int32_t* rowptr, const int32_t* col, const int32_t* nodeJ, const double* nodeq,
                  const int64_t* etab_ptr, const int32_t* edgeJ, const double* edgeq, const int32_t* starts,
                  int32_t num_starts, int64_t num_walks, int32_t walk_length, uint64_t seed, uint32_t walk_id0,
                  int32_t* walks, int32_t* lens, npi_stream_t stream);
int npi_n2v_vocab_count(const int32_t* walks, const int32_t* lens, int64_t num_walks, int32_t walk_length, int32_t V,
                        int64_t* counts, npi_stream_t stream);
int npi_n2v_init_vectors(float* syn0, int64_t V, int32_t dim, uint64_t seed, npi_stream_t stream);
int npi_n2v_skipgram(const int32_t* walks, const int32_t* lens, const int64_t* tok_before, int64_t num_walks,
                     int32_t walk_length, int64_t total_tokens, float* syn0, float* syn1, int32_t V, int32_t dim,
                     const int32_t* negJ, const double* negq, const double* keep, int32_t window, int32_t negative,
                     double alpha, double min_alpha, uint64_t seed, uint32_t walk_id0, int32_t schedule,
                     int32_t max_warps, npi_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Small-subgraph path (csrc/tiny.cu): conv1..3 + pool1..3 + the readout of ONE enclosing subgraph per CTA.
 * Replaces, for batches whose subgraphs have at most npi_tiny_max_nodes() nodes, the per-layer calls of
 * src/classes.py:62-72 (SAGEConv, TopKPooling, cat[gmp, gap], x1 + x2 + x3) and of their backward with ONE launch each
 * (RPI2241's two-hop subgraphs have 15 nodes on average: the layer-by-layer path is launch bound there).  Same buffers,
 * same formulas and the same summation order inside a row as the per-layer entry points; the dense weight gradients
 * (npi_gemm_tn_tc over xp / dxa, npi_gid_reduce + npi_table_grad over dxa[0]) stay separate calls.
 *   graph_ptr[l]   [B+1]: rows of subgraph g at the input layer (l = 0) and after pool l (l = 1..3), npi_batch_prepare.
 *   T, w_label, gid, dist: the virtual input layer -- projected feature table T = table . conv1.weight [V,128], row 0 of
 *                  conv1.weight, global id and hop label per row.
 *   rowptr0 / col0: CSR by destination of the batch (npi_khop_fill).
 *   rowptr_f[l], col_f[l] (l = 0, 1): filtered adjacency after pool l+1, written by the forward and read by the backward:
 *                  subgraph g owns the row pointers rowptr_f[l][graph_ptr[l+1][g] + g ... + n_g] (n_g + 1 of them, so the
 *                  array has N_{l+1} + B + 1 elements) and its entries start at the offset its entries of the layer above
 *                  start at (col_f arrays as long as col0).
 *   weight[l], bias[l], pool_w[l]: conv(l+1).weight (weight[0] is not read), conv(l+1).bias, pool(l+1).weight.
 *   weight_t[l] (l = 1, 2): transposed conv2 / conv3 weights (npi_tiny_transpose), backward only.
 *   h, z, s [N_l], perm / batch [N_{l+1}], new_id [N_l], xp [N_{l+1},128], argmax [B,128]: as in npi_sage_aggregate_fwd,
 *                  npi_topk_select and npi_pool_gate_readout.   y[l] (l = 1, 2): scratch [N_l,128] for the projected rows of layer l+1
 *                  (one buffer per layer: subgraphs are in different layers at the same time).   readout [B,256] is written.
 *   backward: d_readout [B,256]; dpre[l] [N_{l+1},128], dxa[l] [N_l,128] (what the weight-gradient calls read), dxp[l]
 *                  [N_{l+1},128] (l = 0, 1); partials (npi_tiny_partials_bytes(B)); d_pool_w[l] [128], d_bias[l] [128].
 * npi_tiny_bwd phases: 0 = everything, 1 = the per-subgraph kernel (dxa, partials), 2 = d_pool_w / d_bias from the partials.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int32_t B;
    int32_t max_graph_nodes;
    const int32_t* graph_ptr[4];
    const float* T;
    const float* w_label;
    const int32_t* gid;
    const uint8_t* dist;
    const int32_t* rowptr0;
    const int32_t* col0;
    const float* weight[3];
    const float* bias[3];
    const float* pool_w[3];
    const float* weight_t[3];
    float* h[3];
    float* z[3];
    float* s[3];
    int32_t* perm[3];
    int32_t* new_id[3];
    int32_t* batch[3];
    float* xp[3];
    int32_t* argmax[3];
    int32_t* rowptr_f[2];
    int32_t* col_f[2];
    float* y[3];
    float* readout;
    const float* d_readout;
    float* dpre[3];
    float* dxa[3];
    float* dxp[2];
    float* partials;
    float* d_pool_w[3];
    float* d_bias[3];
} npi_tiny_args_t;
int32_t npi_tiny_max_nodes(void);
int64_t npi_tiny_partials_bytes(int32_t B);
int npi_tiny_transpose(const float* w2, const float* w3, float* w2_t, float* w3_t, npi_stream_t stream);
int npi_tiny_fwd(const npi_tiny_args_t* args, npi_stream_t stream);
int npi_tiny_bwd(const npi_tiny_args_t* args, int32_t phases, npi_stream_t stream);
/* The three SAGEConv weight gradients of a small batch in ONE launch, fixed summation order (csrc/tiny.cu):
 *   d conv1.weight [F,128]  = sum_j x_j^T . dxa1_j over the n0 batch rows, x_j = [dist_j | table[gid_j][1:F]] (the virtual
 *                             input row, src/classes.py:706-717) -- the small-batch alternative to npi_gid_reduce +
 *                             npi_table_grad (work proportional to n0 * F instead of V * F);
 *   d conv2.weight [128,128] = x1^T . dxa2 over n1 rows, d conv3.weight = x2^T . dxa3 over n2 rows (x1 / x2: the pooled
 *                             features xp of npi_tiny_fwd; pass x1 = NULL or x2 = NULL to skip a layer) -- the small-batch
 *                             alternative to npi_gemm_tn_tc.
 * The first 1024 bytes of the workspace (ticket counters of the in-kernel reductions) must be zero before the first call;
 * every call leaves them zero. */
int64_t npi_tiny_weight_grads_workspace_bytes(int32_t F);
int npi_tiny_weight_grads(const float* table, int32_t ld, int32_t F, const int32_t* gid, const uint8_t* dist,
                          const float* dxa1, const int32_t* n0_dev, int32_t n0_host, float* d_weight1,
                          const float* x1, const float* dxa2, const int32_t* n1_dev, int32_t n1_host, float* d_weight2,
                          const float* x2, const float* dxa3, const int32_t* n2_dev, int32_t n2_host, float* d_weight3,
                          void* workspace, int64_t workspace_bytes, npi_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NPI_H_ */
